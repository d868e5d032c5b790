"""ctypes binding of liblto_b200.so (include/lto_b200.h).

This is the only way Python reaches the propagation path.  There is no fallback: if the
shared object is missing or no sm_100 device is present the calls raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LTO_B200_LIB") or os.path.join(HERE, "liblto_b200.so")   # LTO_B200_LIB: same override as julia/lto_b200.jl

# src/LowThrustOpt.jl:24-29
MU = 0.012150585609624037
DU = 384747.96285603708
TU = 375699.81732246041
DAY = 86400.0

LTO_FIXED, LTO_ADAPTIVE = 0, 1
LTO_CTRL_RMS, LTO_CTRL_ODE78 = 0, 1
LTO_NORM_STATE, LTO_NORM_STATE_SENS = 0, 1
LTO_KERNEL_AUTO, LTO_KERNEL_GENERIC, LTO_KERNEL_FAST = 0, 1, 2

EXPORTS = [
    "lto_version", "lto_device_count", "lto_init", "lto_init_devices", "lto_n_devices", "lto_destroy", "lto_last_error", "lto_host_alloc", "lto_host_free",
    "lto_kernel_launches", "lto_last_kernel_ms", "lto_stream", "lto_sync", "lto_host_chunk_plan",
    "lto_direct_params_default", "lto_indirect_params_default",
    "lto_direct_defect", "lto_direct_defect_jac", "lto_direct_defect_traj", "lto_direct_defect_jac_traj",
    "lto_indirect_defect", "lto_indirect_defect_jac", "lto_indirect_defect_traj", "lto_indirect_defect_jac_traj",
    "lto_direct_dev", "lto_indirect_dev", "lto_sumsq_dev", "lto_dev_alloc", "lto_dev_free", "lto_ipc_export", "lto_ipc_open", "lto_ipc_close",
    "lto_push_async", "lto_sync_copies", "lto_signal_dev", "lto_wait_dev", "lto_fp64_peak_probe", "lto_debug_profile",
    "lto_indirect_newton", "lto_indirect_newton_dev", "lto_indirect_newton_resolve_dev", "lto_indirect_solve_batch", "lto_direct_qp", "lto_direct_qp_dev", "lto_direct_solve_batch",
    "lto_indirect_newton_nd", "lto_indirect_newton_nd_dev", "lto_indirect_newton_resolve_nd_dev", "lto_indirect_solve_batch_nd",
    "lto_indirect_reduce_fuel_batch", "lto_stack_guess_batch", "lto_indirect_cost_batch", "lto_direct_costates_batch",
    "lto_indirect_switch_batch",
]


class DirectParams(C.Structure):
    _fields_ = [("MU", C.c_double), ("DU", C.c_double), ("TU", C.c_double), ("Isp", C.c_double), ("g0", C.c_double),
                ("default_mass", C.c_double), ("tol", C.c_double), ("mode", C.c_int32), ("err_norm", C.c_int32),
                ("max_attempts", C.c_int32), ("kernel", C.c_int32)]


class IndirectParams(C.Structure):
    _fields_ = [("MU", C.c_double), ("DU", C.c_double), ("TU", C.c_double), ("thrustLimit", C.c_double),
                ("mass", C.c_double), ("time_direction", C.c_double), ("p", C.c_double), ("rho", C.c_double),
                ("Isp", C.c_double), ("g0", C.c_double), ("reltol", C.c_double), ("abstol", C.c_double),
                ("controller", C.c_int32), ("err_norm", C.c_int32), ("max_attempts", C.c_int32), ("kernel", C.c_int32)]


class LtoError(RuntimeError):
    pass


_lib = None


def lib():
    """Load liblto_b200.so; raise loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LtoError("%s is missing: build it with `python -m lowthrustopt_b200.build` "
                           "(there is no non-CUDA implementation of the propagation path)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.lto_last_error.restype = C.c_char_p
        L.lto_last_error.argtypes = [C.c_void_p]
        L.lto_host_alloc.restype = C.c_void_p
        L.lto_host_alloc.argtypes = [C.c_size_t]
        L.lto_host_free.argtypes = [C.c_void_p]
        L.lto_kernel_launches.restype = C.c_int64
        L.lto_kernel_launches.argtypes = [C.c_void_p]
        L.lto_last_kernel_ms.restype = C.c_double
        L.lto_last_kernel_ms.argtypes = [C.c_void_p]
        L.lto_stream.restype = C.c_void_p
        L.lto_stream.argtypes = [C.c_void_p]
        L.lto_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.lto_init_devices.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
        L.lto_n_devices.argtypes = [C.c_void_p]
        L.lto_destroy.argtypes = [C.c_void_p]
        L.lto_sync.argtypes = [C.c_void_p]
        L.lto_host_chunk_plan.argtypes = [C.c_int] * 2 + [C.c_int64] + [C.c_int] * 5 + [C.c_void_p, C.c_int]
        vp, i64, ci = C.c_void_p, C.c_int64, C.c_int
        L.lto_direct_defect.argtypes = [vp, vp, i64, ci, ci] + [vp] * 6 + [vp] * 3
        L.lto_direct_defect_jac.argtypes = [vp, vp, i64, ci, ci] + [vp] * 6 + [vp] * 4
        L.lto_direct_defect_traj.argtypes = [vp, vp, i64, ci, ci, ci] + [vp] * 3 + [vp] * 3
        L.lto_direct_defect_jac_traj.argtypes = [vp, vp, i64, ci, ci, ci] + [vp] * 3 + [vp] * 4
        L.lto_indirect_defect.argtypes = [vp, vp, i64, ci] + [vp] * 6 + [vp] * 3
        L.lto_indirect_defect_jac.argtypes = [vp, vp, i64, ci] + [vp] * 6 + [vp] * 4
        L.lto_indirect_defect_traj.argtypes = [vp, vp, i64, ci, ci] + [vp] * 4 + [vp] * 3
        L.lto_indirect_defect_jac_traj.argtypes = [vp, vp, i64, ci, ci] + [vp] * 4 + [vp] * 4
        L.lto_direct_dev.argtypes = [vp, vp, i64, ci, ci, ci] + [vp] * 6 + [vp] * 4
        L.lto_indirect_dev.argtypes = [vp, vp, i64, ci, ci] + [vp] * 6 + [vp] * 4
        L.lto_sumsq_dev.argtypes = [vp, vp, i64, i64, vp]
        L.lto_dev_alloc.restype = vp
        L.lto_dev_alloc.argtypes = [vp, C.c_size_t]
        L.lto_dev_free.argtypes = [vp, vp]
        L.lto_ipc_export.argtypes = [vp, vp, vp]
        L.lto_ipc_open.argtypes = [vp, vp, C.POINTER(vp)]
        L.lto_ipc_close.argtypes = [vp, vp]
        L.lto_push_async.argtypes = [vp, vp, vp, C.c_size_t]
        L.lto_sync_copies.argtypes = [vp]
        L.lto_signal_dev.argtypes = [vp, vp, C.c_uint64]
        L.lto_wait_dev.argtypes = [vp, vp, C.c_uint64]
        L.lto_fp64_peak_probe.argtypes = [vp, ci, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.lto_debug_profile.argtypes = [vp, vp, ci]
        L.lto_indirect_newton.argtypes = [vp, i64, ci, ci] + [vp] * 4
        L.lto_indirect_newton_dev.argtypes = [vp, i64, ci, ci] + [vp] * 4
        L.lto_indirect_newton_resolve_dev.argtypes = [vp, i64, ci, ci] + [vp] * 3
        L.lto_indirect_solve_batch.argtypes = [vp, vp, i64, ci, ci, ci] + [vp] * 8
        L.lto_indirect_newton_nd.argtypes = [vp, ci, i64, ci, ci] + [vp] * 4
        L.lto_indirect_newton_nd_dev.argtypes = [vp, ci, i64, ci, ci] + [vp] * 4
        L.lto_indirect_newton_resolve_nd_dev.argtypes = [vp, ci, i64, ci, ci] + [vp] * 3
        L.lto_indirect_solve_batch_nd.argtypes = [vp, vp, ci, i64, ci, ci, ci] + [vp] * 8
        L.lto_indirect_reduce_fuel_batch.argtypes = [vp, vp, ci, i64, ci, ci] + [vp] * 11
        L.lto_direct_qp.argtypes = [vp, i64, ci, ci] + [vp] * 9
        L.lto_direct_qp_dev.argtypes = [vp, i64, ci, ci] + [vp] * 9
        L.lto_direct_solve_batch.argtypes = [vp, vp, i64, ci, ci, ci, ci] + [vp] * 5 + [C.c_double] + [vp] * 3
        L.lto_stack_guess_batch.argtypes = [vp, vp, i64, ci, vp, ci, vp, ci] + [vp] * 3 + [vp] * 5
        L.lto_indirect_cost_batch.argtypes = [vp, vp, i64, ci] + [vp] * 4 + [vp] * 4
        L.lto_direct_costates_batch.argtypes = [vp, vp, i64, ci, ci] + [vp] * 5 + [vp] * 4
        L.lto_indirect_switch_batch.argtypes = [vp, vp, i64, ci] + [vp] * 4 + [ci] + [vp] * 6
        _lib = L
    return _lib


def direct_params(Isp=2000.0, mode=LTO_FIXED, tol=1e-13, err_norm=LTO_NORM_STATE, kernel=LTO_KERNEL_AUTO,
                  MU_=MU, DU_=DU, TU_=TU):
    p = DirectParams()
    lib().lto_direct_params_default(C.byref(p))
    p.MU, p.DU, p.TU, p.Isp, p.mode, p.tol, p.err_norm, p.kernel = MU_, DU_, TU_, Isp, mode, tol, err_norm, kernel
    return p


def indirect_params(thrustLimit=0.05, mass=1000.0, time_direction=1.0, p=1.0, rho=1.0, Isp=2000.0, reltol=1e-13,
                    abstol=1e-13, controller=LTO_CTRL_RMS, err_norm=LTO_NORM_STATE_SENS, kernel=LTO_KERNEL_AUTO,
                    MU_=MU, DU_=DU, TU_=TU):
    q = IndirectParams()
    lib().lto_indirect_params_default(C.byref(q))
    q.MU, q.DU, q.TU = MU_, DU_, TU_
    q.thrustLimit, q.mass, q.time_direction, q.p, q.rho, q.Isp = thrustLimit, mass, time_direction, p, rho, Isp
    q.reltol, q.abstol, q.controller, q.err_norm, q.kernel = reltol, abstol, controller, err_norm, kernel
    return q


def host_chunk_plan(method, n_seg, n_nodes=0, nvar=None, nsteps=10, mode=LTO_FIXED, jac=True, n_sm=148):
    """Chunk sizes (segments per launch) of the host-buffer entry points' H2D -> kernel -> D2H pipeline (lto_host_chunk_plan;
    pure host logic, needs no GPU).  method: "direct" | "indirect"."""
    m = {"direct": 0, "indirect": 1}[method]
    nvar = nvar if nvar is not None else (7 if m == 0 else 12)
    buf = (C.c_int64 * 8192)()
    n = lib().lto_host_chunk_plan(m, n_sm, int(n_seg), int(n_nodes), int(nvar), int(nsteps), int(mode), int(bool(jac)), buf, 8192)
    if n < 0:
        raise LtoError("lto_host_chunk_plan: bad arguments (rc %d)" % n)
    return [int(buf[i]) for i in range(min(n, 8192))]


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a)      # raw address (device pointer / pinned buffer)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _shaped(name, a, shape):
    """An input array of exactly `shape` (C-contiguous float64); the C side reads prod(shape) doubles from it unchecked."""
    a = _f64(a)
    if a.shape != tuple(shape):
        raise ValueError("%s must have shape %s (got %s)" % (name, tuple(shape), a.shape))
    return a


def _per_unit(name, a, n):
    """Optional per-segment / per-trajectory parameter array: None, a scalar (broadcast) or exactly (n,) values."""
    if a is None:
        return None
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 0:
        return np.full(n, float(a))
    if a.shape != (n,):
        raise ValueError("%s must be a scalar or have shape (%d,) (got %s)" % (name, n, a.shape))
    return np.ascontiguousarray(a)


def _out(o, key, shape, dtype=np.float64):
    """A caller-supplied output array or a fresh one from the pinned pool; the library writes prod(shape) items into it."""
    a = o.get(key)
    if a is None:
        return _POOL.empty(shape, dtype)
    if not isinstance(a, np.ndarray) or a.dtype != np.dtype(dtype) or a.shape != tuple(shape) or not a.flags["C_CONTIGUOUS"] or not a.flags["WRITEABLE"]:
        raise ValueError("out[%r] must be a writeable C-contiguous %s array of shape %s" % (key, np.dtype(dtype).name, tuple(shape)))
    return a


class PinnedBuffer:
    """Pinned host memory from lto_host_alloc, viewed as a numpy array."""

    def __init__(self, shape, dtype=np.float64):
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = lib().lto_host_alloc(max(nbytes, 1))
        if not self.ptr:
            raise LtoError("lto_host_alloc(%d) failed" % nbytes)
        buf = (C.c_char * max(nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().lto_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _PoolBlock:
    """A pinned block on loan from the pool: goes back when the last numpy view of it is garbage-collected."""
    __slots__ = ("pool", "ptr", "size")

    def __init__(self, pool, ptr, size):
        self.pool, self.ptr, self.size = pool, ptr, size

    def __del__(self):
        try:
            self.pool._give_back(self.ptr, self.size)
        except Exception:
            pass


class PinnedPool:
    """Result arrays of the host-buffer wrappers come out of pinned (page-locked) memory: the device-to-host copy of the Jacobian
    blocks -- 87 % of a config-3 call's bytes -- then runs asynchronously at the PCIe rate and overlaps the kernels, where a copy
    into pageable numpy memory is staged by the driver and serialises the pipeline (bench.py `e2e_pageable`).  cudaHostAlloc is
    expensive (milliseconds), so blocks are recycled: size classes of powers of two, at most `cap_bytes` parked.  This is what
    julia/lto_b200.jl does for the arrays it allocates itself (INTEGRATION.md)."""

    def __init__(self, cap_bytes=2 << 30):
        self.cap, self.parked, self.free = int(cap_bytes), 0, {}

    @staticmethod
    def _cls(nbytes):
        n = 4096
        while n < nbytes:
            n <<= 1
        return n

    def _give_back(self, ptr, size):
        if self.parked + size > self.cap:
            lib().lto_host_free(ptr)
            return
        self.free.setdefault(size, []).append(ptr)
        self.parked += size

    def empty(self, shape, dtype=np.float64):
        shape = tuple(int(x) for x in np.atleast_1d(shape))
        dt = np.dtype(dtype)
        count = int(np.prod(shape, dtype=np.int64))
        nbytes = count * dt.itemsize
        if nbytes == 0:
            return np.empty(shape, dtype=dt)
        size = self._cls(nbytes)
        lst = self.free.get(size)
        if lst:
            ptr = lst.pop(); self.parked -= size
        else:
            ptr = lib().lto_host_alloc(size)
            if not ptr:
                return np.empty(shape, dtype=dt)          # pinned memory exhausted: a pageable array is still correct
        buf = (C.c_char * nbytes).from_address(ptr)
        buf._block = _PoolBlock(self, ptr, size)            # lives as long as any view of the array does
        return np.frombuffer(buf, dtype=dt, count=count).reshape(shape)

    def trim(self):
        for size, lst in self.free.items():
            for ptr in lst:
                lib().lto_host_free(ptr)
        self.free, self.parked = {}, 0


_POOL = PinnedPool()


class Handle:
    """One lto_handle (one CUDA device).  Methods take numpy arrays with one ROW per node /
    segment, i.e. the transpose view of the reference's nstate x n_nodes Julia arrays
    (identical memory)."""

    def __init__(self, device=0):
        """device: an int (lto_init) or a sequence of ints (lto_init_devices: one handle over several GPUs,
        host-buffer entry points only)."""
        self._h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            rc = lib().lto_init_devices(len(device), ids, C.byref(self._h))
        else:
            rc = lib().lto_init(int(device), C.byref(self._h))
        if rc != 0:
            raise LtoError("lto_init(%s) failed (%d): %s" % (device, rc, lib().lto_last_error(None).decode()))
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib().lto_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise LtoError("liblto_b200 error %d: %s" % (rc, lib().lto_last_error(self._h).decode()))

    @property
    def n_devices(self):
        return int(lib().lto_n_devices(self._h))

    @property
    def launches(self):
        return int(lib().lto_kernel_launches(self._h))

    @property
    def last_kernel_ms(self):
        return float(lib().lto_last_kernel_ms(self._h))

    @property
    def stream(self):
        return lib().lto_stream(self._h)

    def sync(self):
        self._ck(lib().lto_sync(self._h))

    def fp64_peak_probe(self, iters=4096):
        f = C.c_double(); ms = C.c_double()
        self._ck(lib().lto_fp64_peak_probe(self._h, int(iters), C.byref(f), C.byref(ms)))
        return f.value, ms.value

    def debug_profile(self, n_words=16384):
        out = np.zeros(n_words, dtype=np.uint64)
        self._ck(lib().lto_debug_profile(self._h, _ptr(out), n_words))
        return out

    # ---- direct ---------------------------------------------------------
    def direct(self, Xa, Xb, ua, ub, ta, tb, nsteps=10, params=None, jac=True, out=None):
        """pairs form.  Xa, Xb: (n_seg, nstate); ua, ub: (n_seg, 3); ta, tb: (n_seg,).
        Returns dict(defect (n_seg,nstate), errors, status, jac (n_seg, 2(nstate+3), nstate) = column-major blocks)."""
        p = params or direct_params()
        Xa = _f64(Xa)
        if Xa.ndim != 2:
            raise ValueError("Xa must be (n_seg, nstate)")
        n_seg, ns = Xa.shape
        Xb = _shaped("Xb", Xb, (n_seg, ns)); ua = _shaped("ua", ua, (n_seg, 3)); ub = _shaped("ub", ub, (n_seg, 3))
        ta = _shaped("ta", ta, (n_seg,)); tb = _shaped("tb", tb, (n_seg,))
        nv = 2 * (ns + 3)
        o = out or {}
        defect = _out(o, "defect", (n_seg, ns)); errors = _out(o, "errors", (n_seg,))
        status = _out(o, "status", (n_seg,), np.int32)
        if jac:
            J = _out(o, "jac", (n_seg, nv, ns))
            self._ck(lib().lto_direct_defect_jac(self._h, C.addressof(p), n_seg, ns, int(nsteps), _ptr(Xa), _ptr(Xb), _ptr(ua),
                                                 _ptr(ub), _ptr(ta), _ptr(tb), _ptr(defect), _ptr(errors), _ptr(status), _ptr(J)))
            return dict(defect=defect, errors=errors, status=status, jac=J)
        self._ck(lib().lto_direct_defect(self._h, C.addressof(p), n_seg, ns, int(nsteps), _ptr(Xa), _ptr(Xb), _ptr(ua), _ptr(ub),
                                         _ptr(ta), _ptr(tb), _ptr(defect), _ptr(errors), _ptr(status)))
        return dict(defect=defect, errors=errors, status=status)

    def direct_traj(self, X_all, u_all, t_TU, nsteps=10, params=None, jac=True):
        """trajectory form.  X_all: (n_traj, n_nodes, nstate) (or (n_nodes, nstate)), u_all: (.., n_nodes, 3), t_TU: (.., n_nodes)."""
        p = params or direct_params()
        X_all, u_all, t_TU = map(_f64, (X_all, u_all, t_TU))
        if X_all.ndim == 2:
            X_all, u_all, t_TU = X_all[None], u_all[None], t_TU[None]
        if X_all.ndim != 3:
            raise ValueError("X_all must be (n_traj, n_nodes, nstate)")
        n_traj, n_nodes, ns = X_all.shape
        u_all = _shaped("u_all", u_all, (n_traj, n_nodes, 3)); t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        n_seg = n_traj * (n_nodes - 1); nv = 2 * (ns + 3)
        defect = _POOL.empty((n_seg, ns)); errors = _POOL.empty((n_seg,)); status = _POOL.empty((n_seg,), np.int32)
        if jac:
            J = _POOL.empty((n_seg, nv, ns))
            self._ck(lib().lto_direct_defect_jac_traj(self._h, C.addressof(p), n_traj, n_nodes, ns, int(nsteps), _ptr(X_all),
                                                      _ptr(u_all), _ptr(t_TU), _ptr(defect), _ptr(errors), _ptr(status), _ptr(J)))
            return dict(defect=defect, errors=errors, status=status, jac=J)
        self._ck(lib().lto_direct_defect_traj(self._h, C.addressof(p), n_traj, n_nodes, ns, int(nsteps), _ptr(X_all), _ptr(u_all),
                                              _ptr(t_TU), _ptr(defect), _ptr(errors), _ptr(status)))
        return dict(defect=defect, errors=errors, status=status)

    # ---- indirect -------------------------------------------------------
    def indirect(self, x0, t0, t1, x_target=None, params=None, thrustLimit=None, rho=None, jac=True, out=None):
        """pairs form.  x0: (n_seg, ndim).  Returns dict(defect, status, nsteps (n_seg,2), phi (n_seg, ndim, ndim) column-major).
        `out` may supply preallocated (e.g. pinned) arrays under the same keys."""
        p = params or indirect_params()
        x0 = _f64(x0)
        if x0.ndim != 2:
            raise ValueError("x0 must be (n_seg, ndim)")
        n_seg, nd = x0.shape
        t0 = _shaped("t0", t0, (n_seg,)); t1 = _shaped("t1", t1, (n_seg,))
        xt = None if x_target is None else _shaped("x_target", x_target, (n_seg, nd))
        tl = _per_unit("thrustLimit", thrustLimit, n_seg)
        rh = _per_unit("rho", rho, n_seg)
        o = out or {}
        defect = _out(o, "defect", (n_seg, nd)); status = _out(o, "status", (n_seg,), np.int32)
        nst = _out(o, "nsteps", (n_seg, 2), np.int32)
        if jac:
            phi = _out(o, "phi", (n_seg, nd, nd))
            self._ck(lib().lto_indirect_defect_jac(self._h, C.addressof(p), n_seg, nd, _ptr(x0), _ptr(t0), _ptr(t1), _ptr(xt),
                                                   _ptr(tl), _ptr(rh), _ptr(defect), _ptr(status), _ptr(nst), _ptr(phi)))
            return dict(defect=defect, status=status, nsteps=nst, phi=phi)
        self._ck(lib().lto_indirect_defect(self._h, C.addressof(p), n_seg, nd, _ptr(x0), _ptr(t0), _ptr(t1), _ptr(xt), _ptr(tl),
                                           _ptr(rh), _ptr(defect), _ptr(status), _ptr(nst)))
        return dict(defect=defect, status=status, nsteps=nst)

    def indirect_traj(self, XC_all, t_TU, params=None, thrustLimit=None, rho=None, jac=True):
        """trajectory form.  XC_all: (n_traj, n_nodes, ndim) or (n_nodes, ndim); thrustLimit/rho: optional (n_traj,)."""
        p = params or indirect_params()
        XC_all, t_TU = _f64(XC_all), _f64(t_TU)
        if XC_all.ndim == 2:
            XC_all, t_TU = XC_all[None], t_TU[None]
        if XC_all.ndim != 3:
            raise ValueError("XC_all must be (n_traj, n_nodes, ndim)")
        n_traj, n_nodes, nd = XC_all.shape
        t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        n_seg = n_traj * (n_nodes - 1)
        tl = _per_unit("thrustLimit", thrustLimit, n_traj)
        rh = _per_unit("rho", rho, n_traj)
        defect = _POOL.empty((n_seg, nd)); status = _POOL.empty((n_seg,), np.int32); nst = _POOL.empty((n_seg, 2), np.int32)
        if jac:
            phi = _POOL.empty((n_seg, nd, nd))
            self._ck(lib().lto_indirect_defect_jac_traj(self._h, C.addressof(p), n_traj, n_nodes, nd, _ptr(XC_all), _ptr(t_TU),
                                                        _ptr(tl), _ptr(rh), _ptr(defect), _ptr(status), _ptr(nst), _ptr(phi)))
            return dict(defect=defect, status=status, nsteps=nst, phi=phi)
        self._ck(lib().lto_indirect_defect_traj(self._h, C.addressof(p), n_traj, n_nodes, nd, _ptr(XC_all), _ptr(t_TU), _ptr(tl),
                                                _ptr(rh), _ptr(defect), _ptr(status), _ptr(nst)))
        return dict(defect=defect, status=status, nsteps=nst)

    def indirect_cost_batch(self, XC_all, t_TU, params=None, thrustLimit=None, rho=None, defect=False):
        """Control cost of 12-dim indirect trajectories in one device call (lto_indirect_cost_batch): the defect-only kernel's steps with
        the quadratures of |a_u| and |a_u|^2 on them.  XC_all: (n_traj, n_nodes, 12); t_TU: (n_traj, n_nodes), finite and non-decreasing;
        thrustLimit / rho: scalars or (n_traj,); params.controller must be LTO_CTRL_RMS.  defect: also return the defects (bitwise those of
        indirect_traj(jac=False)).  Returns dict(dv (m/s), energy (N^2 TU), status (worst segment status)[, defect (n_traj, n_nodes-1, 12)])."""
        p = params or indirect_params()
        XC = _f64(XC_all)
        if XC.ndim != 3 or XC.shape[2] != 12:
            raise ValueError("XC_all must be (n_traj, n_nodes, 12): the cost quadrature is in the 12-dim kernel (got %s)" % (XC.shape,))
        n_traj, n_nodes, _ = XC.shape
        if n_nodes < 2:
            raise ValueError("n_nodes must be >= 2 (got %d)" % n_nodes)
        if p.controller != LTO_CTRL_RMS:
            raise ValueError("the cost quadrature needs controller = LTO_CTRL_RMS (got %d)" % p.controller)
        t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        bad = ~np.isfinite(t_TU).all(axis=1) | (np.diff(t_TU, axis=1) < 0).any(axis=1)
        if bad.any():
            raise ValueError("trajectory %d: t_TU must be finite and non-decreasing (reversed spans are not supported)" % int(np.argmax(bad)))
        tl = _per_unit("thrustLimit", thrustLimit, n_traj)
        rh = _per_unit("rho", rho, n_traj)
        dv = np.empty(n_traj); energy = np.empty(n_traj); status = np.empty(n_traj, dtype=np.int32)
        d = np.empty((n_traj, n_nodes - 1, 12)) if defect else None
        self._ck(lib().lto_indirect_cost_batch(self._h, C.addressof(p), n_traj, n_nodes, _ptr(XC), _ptr(t_TU), _ptr(tl), _ptr(rh), _ptr(dv),
                                               _ptr(energy), _ptr(d), _ptr(status)))
        out = dict(dv=dv, energy=energy, status=status)
        if defect:
            out["defect"] = d
        return out

    def indirect_switch_batch(self, XC_all, t_TU, params=None, thrustLimit=None, rho=None, max_switch=16, defect=False):
        """Switch times of 12-dim p = 1 indirect trajectories in one device call (lto_indirect_switch_batch): the sign changes of
        S = |lv| - 1 (thrust on where S > 0), located on the defect-only kernel's steps, with one switch at a node where the propagated end of
        the segment before it and the node lie on opposite sides.  XC_all: (n_traj, n_nodes, 12); t_TU: (n_traj, n_nodes), finite and
        non-decreasing; thrustLimit / rho: scalars or (n_traj,); params.p must be 1 and params.controller LTO_CTRL_RMS; max_switch in
        [1, 64].  defect: also return the defects (bitwise those of indirect_traj(jac=False)).
        Returns dict(t_switch (n_traj, max_switch) in TU, NaN in unused slots; direction (n_traj, max_switch): +1 a burn starts, -1 it ends,
        0 unused; n_switch (n_traj,): the true count (> max_switch: truncated; -1 where status is not LTO_ST_OK); on_start (n_traj,);
        status (n_traj,)[, defect (n_traj, n_nodes-1, 12)])."""
        p = params or indirect_params()
        XC = _f64(XC_all)
        if XC.ndim != 3 or XC.shape[2] != 12:
            raise ValueError("XC_all must be (n_traj, n_nodes, 12): the switch scan is in the 12-dim kernel (got %s)" % (XC.shape,))
        n_traj, n_nodes, _ = XC.shape
        if n_nodes < 2:
            raise ValueError("n_nodes must be >= 2 (got %d)" % n_nodes)
        if p.controller != LTO_CTRL_RMS:
            raise ValueError("the switch scan needs controller = LTO_CTRL_RMS (got %d)" % p.controller)
        if p.p != 1.0:
            raise ValueError("switch times are defined for the p = 1 law only (got p = %g)" % p.p)
        if not (isinstance(max_switch, (int, np.integer)) and 1 <= max_switch <= 64):
            raise ValueError("max_switch must be an integer in [1, 64] (got %r)" % (max_switch,))
        t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        bad = ~np.isfinite(t_TU).all(axis=1) | (np.diff(t_TU, axis=1) < 0).any(axis=1)
        if bad.any():
            raise ValueError("trajectory %d: t_TU must be finite and non-decreasing (reversed spans are not supported)" % int(np.argmax(bad)))
        tl = _per_unit("thrustLimit", thrustLimit, n_traj)
        rh = _per_unit("rho", rho, n_traj)
        K = int(max_switch)
        ts = np.empty((n_traj, K)); dr = np.empty((n_traj, K), dtype=np.int32)
        ns = np.empty(n_traj, dtype=np.int32); on = np.empty(n_traj, dtype=np.int32); status = np.empty(n_traj, dtype=np.int32)
        d = np.empty((n_traj, n_nodes - 1, 12)) if defect else None
        self._ck(lib().lto_indirect_switch_batch(self._h, C.addressof(p), n_traj, n_nodes, _ptr(XC), _ptr(t_TU), _ptr(tl), _ptr(rh), K,
                                                 _ptr(ts), _ptr(dr), _ptr(ns), _ptr(on), _ptr(d), _ptr(status)))
        out = dict(t_switch=ts, direction=dr, n_switch=ns, on_start=on, status=status)
        if defect:
            out["defect"] = d
        return out

    # ---- device-resident (raw device addresses, e.g. torch .data_ptr()) --
    def direct_dev(self, params, n_seg, n_nodes, nstate, nsteps, Xa, Xb, ua, ub, ta, tb, defect, errors, status, jac):
        self._ck(lib().lto_direct_dev(self._h, C.addressof(params), int(n_seg), int(n_nodes), int(nstate), int(nsteps), _ptr(Xa),
                                      _ptr(Xb), _ptr(ua), _ptr(ub), _ptr(ta), _ptr(tb), _ptr(defect), _ptr(errors), _ptr(status),
                                      _ptr(jac)))

    # ---- peer memory --------------------------------------------------
    def dev_alloc(self, nbytes):
        p = lib().lto_dev_alloc(self._h, int(nbytes))
        if not p:
            raise LtoError("lto_dev_alloc(%d) failed: %s" % (nbytes, lib().lto_last_error(self._h).decode()))
        return int(p)

    def dev_free(self, ptr):
        lib().lto_dev_free(self._h, C.c_void_p(ptr))

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        self._ck(lib().lto_ipc_export(self._h, C.c_void_p(ptr), buf))
        return bytes(buf.raw)

    def ipc_open(self, handle64):
        out = C.c_void_p()
        self._ck(lib().lto_ipc_open(self._h, C.create_string_buffer(handle64, 64), C.byref(out)))
        return int(out.value)

    def ipc_close(self, ptr):
        self._ck(lib().lto_ipc_close(self._h, C.c_void_p(ptr)))

    def push_async(self, dst, src, nbytes):
        self._ck(lib().lto_push_async(self._h, C.c_void_p(dst), C.c_void_p(src), int(nbytes)))

    def sync_copies(self):
        self._ck(lib().lto_sync_copies(self._h))

    def signal_dev(self, flag_ptr, value):
        self._ck(lib().lto_signal_dev(self._h, C.c_void_p(flag_ptr), int(value)))

    def wait_dev(self, flag_ptr, value):
        self._ck(lib().lto_wait_dev(self._h, C.c_void_p(flag_ptr), int(value)))

    def sumsq_dev(self, v, n_rows, row_len, out):
        self._ck(lib().lto_sumsq_dev(self._h, _ptr(v), int(n_rows), int(row_len), _ptr(out)))

    def indirect_dev(self, params, n_seg, n_nodes, ndim, x0, t0, t1, x_target, thrustLimit, rho, defect, status, nsteps_out, phi):
        self._ck(lib().lto_indirect_dev(self._h, C.addressof(params), int(n_seg), int(n_nodes), int(ndim), _ptr(x0), _ptr(t0),
                                        _ptr(t1), _ptr(x_target), _ptr(thrustLimit), _ptr(rho), _ptr(defect), _ptr(status),
                                        _ptr(nsteps_out), _ptr(phi)))

    # ---- Newton update / batched solver of the indirect method (device side) ----
    def indirect_newton(self, phi, defect, flag_adjointsOnly=False):
        """xc_update = -sparse(Jac_full) \\ defect_vec (multiShoot_CRTBP_indirect.jl:181-182) for a batch of trajectories.
        phi: (n_traj, n_nodes-1, m, m) column-major blocks as the propagation returns them ([.., col, row]), m = 12 or 14 (the
        14-dim system with mass; end pins in include/lto_b200.h); defect: (n_traj, n_nodes-1, m).
        Returns (xc_update (n_traj, n_nodes, m), status (n_traj,))."""
        phi, defect = _f64(phi), _f64(defect)
        if phi.ndim == 3:
            phi, defect = phi[None], defect[None]
        if phi.ndim != 4:
            raise ValueError("phi must be (n_traj, n_nodes-1, m, m) with m = 12 or 14")
        n_traj, nseg, m, m2 = phi.shape
        if m not in (12, 14) or m2 != m or defect.shape != (n_traj, nseg, m):
            raise ValueError("phi must be (n_traj, n_nodes-1, m, m) and defect (n_traj, n_nodes-1, m) with m = 12 or 14 "
                             "(got phi %s, defect %s)" % (phi.shape, defect.shape))
        upd = np.empty((n_traj, nseg + 1, m)); status = np.empty(n_traj, dtype=np.int32)
        self._ck(lib().lto_indirect_newton_nd(self._h, m, n_traj, nseg + 1, int(bool(flag_adjointsOnly)), _ptr(phi), _ptr(defect), _ptr(upd),
                                              _ptr(status)))
        return upd, status

    def indirect_newton_dev(self, n_traj, n_nodes, flag_adjointsOnly, phi, defect, xc_update, status=None, ndim=12):
        self._ck(lib().lto_indirect_newton_nd_dev(self._h, int(ndim), int(n_traj), int(n_nodes), int(bool(flag_adjointsOnly)), _ptr(phi),
                                                  _ptr(defect), _ptr(xc_update), _ptr(status)))

    def indirect_newton_resolve_dev(self, n_traj, n_nodes, flag_adjointsOnly, defect, xc_update, status=None, ndim=12):
        """Same matrix as the preceding indirect_newton_dev call (same shape, mode and ndim), new defects (the second-order correction, :207)."""
        self._ck(lib().lto_indirect_newton_resolve_nd_dev(self._h, int(ndim), int(n_traj), int(n_nodes), int(bool(flag_adjointsOnly)),
                                                          _ptr(defect), _ptr(xc_update), _ptr(status)))

    def indirect_solve_batch(self, XC_all, t_TU, params=None, thrustLimit=None, rho=None, max_iter=50, flag_adjointsOnly=False, inplace=False,
                             out=None):
        """multiShoot_CRTBP_indirect (:58-345) for n_traj trajectories at once, iterated on the device.
        XC_all: (n_traj, n_nodes, m), m = 12 (the reference's system) or 14 ([r v m | lr lv lm], params.Isp in the mass flow; end pins
        in include/lto_b200.h); t_TU: (n_traj, n_nodes).  Returns dict(XC_all, defect, status_flag, iters, er).
        inplace: work directly on XC_all (must be a C-contiguous float64 array, e.g. pinned) as the C entry point does;
        out: optional preallocated arrays under the keys defect / status_flag / iters / er."""
        p = params or indirect_params()
        if inplace:
            XC = XC_all
            if not (isinstance(XC, np.ndarray) and XC.dtype == np.float64 and XC.flags.c_contiguous):
                raise ValueError("inplace needs a C-contiguous float64 array")
        else:
            XC = np.array(XC_all, dtype=np.float64, order="C")
        t_TU = _f64(t_TU)
        if XC.ndim == 2:
            XC, t_TU = XC[None], t_TU[None]
        n_traj, n_nodes, nd = XC.shape
        if nd not in (12, 14):
            raise ValueError("XC_all must have 12 (the reference's system, multiShoot_CRTBP_indirect.jl:258) or 14 columns (got %d)" % nd)
        t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        tl = _per_unit("thrustLimit", thrustLimit, n_traj)
        rh = _per_unit("rho", rho, n_traj)
        o = out or {}
        defect = _out(o, "defect", (n_traj, n_nodes - 1, nd))
        flag = _out(o, "status_flag", (n_traj,), np.int32)
        iters = _out(o, "iters", (n_traj,), np.int32)
        er = _out(o, "er", (n_traj,))
        self._ck(lib().lto_indirect_solve_batch_nd(self._h, C.addressof(p), nd, n_traj, n_nodes, int(max_iter), int(bool(flag_adjointsOnly)),
                                                   _ptr(XC), _ptr(t_TU), _ptr(tl), _ptr(rh), _ptr(defect), _ptr(flag), _ptr(iters), _ptr(er)))
        return dict(XC_all=XC, defect=defect, status_flag=flag, iters=iters, er=er)

    def indirect_reduce_fuel_batch(self, XC_all, t_TU, rho_current, rho_target, backoff_uniform, params=None, thrustLimit=None, max_iter=10):
        """reduceFuel_indirect (HelperFunctions.jl:105-193) for n_traj independent rho ladders in one call, every solver call and the
        ladder logic on the device (lto_indirect_reduce_fuel_batch).  XC_all: (n_traj, n_nodes, m), m = 12 or 14; t_TU: (n_traj, n_nodes);
        rho_current, rho_target, thrustLimit: scalars or (n_traj,); backoff_uniform: (n_traj, 100) draws in [0, 1) for the back-off
        rho *= 3(1 + u) (:182), consumed in order; params.p must be 1; max_iter: maxIter of every solver call.
        Returns dict(XC_all, defect, status (3: gave up after 100 rungs), calls, newton_iters, rho_last)."""
        p = params or indirect_params()
        XC = np.array(XC_all, dtype=np.float64, order="C")
        if XC.ndim != 3 or XC.shape[2] not in (12, 14):
            raise ValueError("XC_all must be (n_traj, n_nodes, 12 or 14) (got %s)" % (XC.shape,))
        n_traj, n_nodes, nd = XC.shape
        t_TU = _shaped("t_TU", t_TU, (n_traj, n_nodes))
        r0 = _per_unit("rho_current", rho_current, n_traj); r1 = _per_unit("rho_target", rho_target, n_traj)
        tl = _per_unit("thrustLimit", thrustLimit, n_traj)
        draws = _shaped("backoff_uniform", backoff_uniform, (n_traj, 100))
        defect = np.empty((n_traj, n_nodes - 1, nd)); status = np.empty(n_traj, dtype=np.int32)
        calls = np.empty(n_traj, dtype=np.int32); nit = np.empty(n_traj, dtype=np.int32); rho_last = np.empty(n_traj)
        self._ck(lib().lto_indirect_reduce_fuel_batch(self._h, C.addressof(p), nd, n_traj, n_nodes, int(max_iter), _ptr(XC), _ptr(t_TU), _ptr(tl),
                                                      _ptr(r0), _ptr(r1), _ptr(draws), _ptr(defect), _ptr(status), _ptr(calls), _ptr(nit),
                                                      _ptr(rho_last)))
        return dict(XC_all=XC, defect=defect, status=status, calls=calls, newton_iters=nit, rho_last=rho_last)

    # ---- direct method: the QP of optimizeTraj on the device ----
    def direct_qp(self, jac, defect, u_all, t_TU, b0, bf):
        """optimizeTraj's linear subproblem (multiShoot_CRTBP_direct.jl:248-403, flagEnd = false, allowImpulsive = false) for a batch.
        jac: (n_traj, n_nodes-1, 2(n+3), n) column-major blocks as direct_traj returns them; defect: (n_traj, n_nodes-1, n);
        u_all: (n_traj, n_nodes, 3); t_TU: (n_traj, n_nodes); b0: (n_traj, 6 or 7); bf: (n_traj, 6).
        Returns (x_update (n_traj, n_nodes, n), u_update (n_traj, n_nodes, 3), status (n_traj,))."""
        jac, defect, u_all, t_TU, b0, bf = map(_f64, (jac, defect, u_all, t_TU, b0, bf))
        n_traj, nseg, nv, n = jac.shape
        N = nseg + 1
        if nv != 2 * (n + 3) or defect.shape != (n_traj, nseg, n) or u_all.shape != (n_traj, N, 3) or t_TU.shape != (n_traj, N):
            raise ValueError("inconsistent shapes")
        if b0.shape != (n_traj, 6 + (n == 7)) or bf.shape != (n_traj, 6):
            raise ValueError("b0 must be (n_traj, 6 or 7) and bf (n_traj, 6)")
        xu = np.empty((n_traj, N, n)); uu = np.empty((n_traj, N, 3)); status = np.empty(n_traj, dtype=np.int32)
        self._ck(lib().lto_direct_qp(self._h, n_traj, N, n, _ptr(jac), _ptr(defect), _ptr(u_all), _ptr(t_TU), _ptr(b0), _ptr(bf), _ptr(xu), _ptr(uu),
                                     _ptr(status)))
        return xu, uu, status

    def direct_solve_batch(self, X_all, u_all, t_TU, state_0, state_f, mass=1000.0, nsteps=10, max_iter=100, params=None):
        """multiShoot_CRTBP_direct (:465-594, the demo's setting) for n_traj trajectories at once, iterated on the device.
        X_all: (n_traj, n_nodes, nstate); u_all: (n_traj, n_nodes, 3); t_TU: (n_traj, n_nodes); state_0, state_f: (n_traj, 6).
        Returns dict(X_all, u_all, defect, iters, er)."""
        p = params or direct_params()
        X = np.array(X_all, dtype=np.float64, order="C"); U = np.array(u_all, dtype=np.float64, order="C")
        t_TU, state_0, state_f = map(_f64, (t_TU, state_0, state_f))
        n_traj, n_nodes, ns = X.shape
        if U.shape != (n_traj, n_nodes, 3) or t_TU.shape != (n_traj, n_nodes) or state_0.shape != (n_traj, 6) or state_f.shape != (n_traj, 6):
            raise ValueError("inconsistent shapes")
        defect = np.empty((n_traj, n_nodes - 1, ns)); iters = np.empty(n_traj, dtype=np.int32); er = np.empty(n_traj)
        self._ck(lib().lto_direct_solve_batch(self._h, C.addressof(p), n_traj, n_nodes, ns, int(nsteps), int(max_iter), _ptr(X), _ptr(U), _ptr(t_TU),
                                              _ptr(state_0), _ptr(state_f), float(mass), _ptr(defect), _ptr(iters), _ptr(er)))
        return dict(X_all=X, u_all=U, defect=defect, iters=iters, er=er)

    def direct_costates_batch(self, X, U, t, state_0, state_f, nsteps=10, params=None):
        """Costates of nstate-6 direct solutions from the dual solution of optimizeTraj's QP (lto_direct_costates_batch): K1's Jacobian
        blocks at (X, U), then K7's multipliers of the defect rows mapped to the node costates of the 12-dim p = 2 system.
        X: (n_traj, n_nodes, 6); U: (n_traj, n_nodes, 3); t: (n_traj, n_nodes), finite and strictly increasing; state_0, state_f: (n_traj, 6);
        params.mode must be LTO_FIXED.  Returns dict(XC_all (n_traj, n_nodes, 12): X bitwise and the costates (NaN where status != 0),
        multipliers (n_traj, n_nodes-1, 6), du_max (n_traj,): max |du| in N of the QP step at (X, U), status (n_traj,))."""
        p = params or direct_params()
        X = _f64(X)
        if X.ndim != 3 or X.shape[2] != 6:
            raise ValueError("X must be (n_traj, n_nodes, 6): the costate map is for nstate 6 (got %s)" % (X.shape,))
        n_traj, n_nodes, _ = X.shape
        if n_nodes < 2:
            raise ValueError("n_nodes must be >= 2 (got %d)" % n_nodes)
        if p.mode != LTO_FIXED:
            raise ValueError("the direct costates run the fixed-grid path: params.mode must be LTO_FIXED (got %d)" % p.mode)
        U = _shaped("U", U, (n_traj, n_nodes, 3)); t = _shaped("t", t, (n_traj, n_nodes))
        state_0 = _shaped("state_0", state_0, (n_traj, 6)); state_f = _shaped("state_f", state_f, (n_traj, 6))
        bad = ~np.isfinite(t).all(axis=1) | ~(np.diff(t, axis=1) > 0).all(axis=1)
        if bad.any():
            raise ValueError("trajectory %d: t must be finite and strictly increasing" % int(np.argmax(bad)))
        XC = np.empty((n_traj, n_nodes, 12)); mult = np.empty((n_traj, n_nodes - 1, 6)); du = np.empty(n_traj)
        status = np.empty(n_traj, dtype=np.int32)
        self._ck(lib().lto_direct_costates_batch(self._h, C.addressof(p), n_traj, n_nodes, int(nsteps), _ptr(X), _ptr(U), _ptr(t), _ptr(state_0),
                                                 _ptr(state_f), _ptr(XC), _ptr(mult), _ptr(du), _ptr(status)))
        return dict(XC_all=XC, multipliers=mult, du_max=du, status=status)

    # ---- the trajectory-stacking initial guess on the device ----
    def stack_guess_batch(self, X0_states, Xf_states, tau1, t_TU, t_split, params=None):
        """The demos' trajectory-stacking guess (CRTBP_Multishoot_direct_demo.jl:117-157, solvers.trajectory_stack_guess) for n_traj
        transfers in one device call (lto_stack_guess_batch).  X0_states, Xf_states: the reference's (6, n) orbit tables; tau1, t_split:
        (n_traj,); t_TU: (n_traj, n_nodes).  params: the arcs' indirect parameters, by default the host mirror's
        (thrustLimit 0, mass 1e3, p = rho = 1).
        Returns dict(XC_all (n_traj, n_nodes, 12), tau2 (n_traj,), state_0 (n_traj, 6), state_f (n_traj, 6), status (n_traj,))."""
        p = params or indirect_params(thrustLimit=0.0, mass=1e3, time_direction=1.0, p=1.0, rho=1.0)
        X0, Xf = _f64(X0_states), _f64(Xf_states)
        if X0.ndim != 2 or X0.shape[0] != 6 or Xf.ndim != 2 or Xf.shape[0] != 6:
            raise ValueError("X0_states and Xf_states must be (6, n) orbit tables (got %s, %s)" % (X0.shape, Xf.shape))
        t_TU = _f64(t_TU)
        if t_TU.ndim != 2:
            raise ValueError("t_TU must be (n_traj, n_nodes) (got %s)" % (t_TU.shape,))
        n_traj, n_nodes = t_TU.shape
        tau1 = _shaped("tau1", tau1, (n_traj,)); t_split = _shaped("t_split", t_split, (n_traj,))
        X0c, Xfc = np.ascontiguousarray(X0.T), np.ascontiguousarray(Xf.T)                # column-major 6 x n
        XC = np.empty((n_traj, n_nodes, 12)); tau2 = np.empty(n_traj); s0 = np.empty((n_traj, 6)); sf = np.empty((n_traj, 6))
        status = np.empty(n_traj, dtype=np.int32)
        self._ck(lib().lto_stack_guess_batch(self._h, C.addressof(p), n_traj, n_nodes, _ptr(X0c), X0.shape[1], _ptr(Xfc), Xf.shape[1], _ptr(tau1),
                                             _ptr(t_TU), _ptr(t_split), _ptr(XC), _ptr(tau2), _ptr(s0), _ptr(sf), _ptr(status)))
        return dict(XC_all=XC, tau2=tau2, state_0=s0, state_f=sf, status=status)
