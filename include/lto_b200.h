/* lto_b200.h -- C ABI of liblto_b200.so: B200 (sm_100a) segment propagation for
 * LowThrustOpt's multiple-shooting solvers.
 *
 * The library replaces, and only replaces, the four inner closures of the reference
 * (citations relative to the reference repository root):
 *
 *   direct   defectCalc    src/multiShoot_CRTBP_direct.jl:66-109    -> lto_direct_defect[_traj]
 *   direct   jacobianCalc  src/multiShoot_CRTBP_direct.jl:111-143   -> lto_direct_defect_jac[_traj]
 *            (the dense Jac_temp blocks; the band scatter :146-162 stays on the host)
 *   indirect defectCalc    src/multiShoot_CRTBP_indirect.jl:63-90   -> lto_indirect_defect[_traj]
 *   indirect jacobianCalc  src/multiShoot_CRTBP_indirect.jl:93-124  -> lto_indirect_defect_jac[_traj]
 *            (the Phi_i blocks of hcat(Phi_i, -I) :123; scatter/pinning :128-142 stay on the host)
 *
 * and beneath them the integrator hooks  ode7_8 (GeneralCode/ode.jl:773-953),
 * ode78 (GeneralCode/ode.jl:364-544), solve(prob, Vern8(), reltol, abstol)
 * (multiShoot_CRTBP_indirect.jl:78-79,107-110) and ForwardDiff.jacobian (:121), with the
 * right-hand sides CRTBP_prop_EP_deriv (src/CRTBP_prop_EP_deriv.jl:8-61) and
 * CRTBP_stateCostate_deriv! (src/CRTBP_stateCostate_deriv.jl:9-90) compiled in.
 *
 * Conventions
 *  - All arrays are Float64, laid out exactly as Julia lays out the reference's
 *    arrays (column-major): X_all is nstate x n_nodes, so node i's state is the
 *    contiguous run X_all + i*nstate.  "pairs" entry points take one row of
 *    (a, b) node data per segment in the same per-node layout.
 *  - Caller owns every buffer; nothing is retained after return.  Buffers may be
 *    ordinary (pageable) memory or memory from lto_host_alloc (pinned: faster copies).
 *  - Return value: 0 ok, negative = library failure (see lto_last_error).  Numerical
 *    trouble is per segment in status[] (LTO_ST_*), never a failure.
 *  - A handle is bound to one CUDA device (lto_init) or a fixed set (lto_init_devices) and is not re-entrant.
 *  - There is no CPU fallback: without a usable sm_100 device lto_init fails.
 */
#ifndef LTO_B200_H
#define LTO_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTO_B200_VERSION 100

/* per-segment status codes */
/* Time spans: every indirect segment is integrated FORWARDS from t0 to t1.  t1 == t0 is allowed (returns x0 and Phi = I).  t1 < t0
 * (the reference's ODEProblem would integrate backwards) is NOT supported: the host-buffer entry points refuse the call with
 * LTO_ERR_ARG naming the first such segment; the device-pointer entry points (lto_indirect_dev, the batched solver) cannot look at
 * the times and treat such a segment as an empty span -- callers of those must not pass reversed spans.  time_direction = -1 in the
 * parameters (the backward legs of the reference's direct method and of its trajectory stacking) is the supported way of
 * integrating the time-reversed dynamics.  The host-buffer entry points also refuse a NaN or infinite t0 / t1; the device-pointer
 * entry points still do not look at the times (the generic kernel reports such a segment as LTO_ST_NAN, or LTO_ST_HMIN when reversed).
 * Direct segments (both legs run from ta to t_mid = ta + (tb - ta) / 2), every entry point and kernel:
 *   - a NaN or infinite ta / tb gives LTO_ST_NAN;
 *   - tb == ta gives LTO_ST_OK with zero-length legs;
 *   - tb < ta: LTO_FIXED integrates the legs backwards on the same grid (what the reference's ode7_8 does), status LTO_ST_OK;
 *     LTO_ADAPTIVE does not integrate such a leg and gives LTO_ST_HMIN. */
enum { LTO_ST_OK = 0, LTO_ST_NAN = 1, LTO_ST_HMIN = 2, LTO_ST_MAXSTEPS = 3, LTO_ST_BADP = 4 };
/* return codes */
enum { LTO_SUCCESS = 0, LTO_ERR_CUDA = -1, LTO_ERR_ARG = -2, LTO_ERR_NODEVICE = -3, LTO_ERR_NOMEM = -4 };
/* direct integration mode */
enum { LTO_FIXED = 0,      /* ode7_8: fixed grid LinRange(t_i, t_mid, nsteps) -- what the reference runs */
       LTO_ADAPTIVE = 1 }; /* ode78 controller (ode.jl:477-534) on every leg */
/* indirect controller */
enum { LTO_CTRL_RMS = 0,   /* OrdinaryDiffEq-style: scaled RMS error, reltol/abstol (stands in for Vern8) */
       LTO_CTRL_ODE78 = 1 };/* the reference's own ode78 controller, tol = reltol */
/* which components the step-size controller's norms span */
enum { LTO_NORM_STATE = 0, LTO_NORM_STATE_SENS = 1 };
/* kernel selection */
enum { LTO_KERNEL_AUTO = 0, LTO_KERNEL_GENERIC = 1, LTO_KERNEL_FAST = 2 };

typedef struct lto_handle lto_handle;

/* Free variables / arguments of the direct closures (multiShoot_CRTBP_direct.jl:66,86). */
typedef struct lto_direct_params {
    double MU, DU, TU;     /* src/LowThrustOpt.jl:24-26 */
    double Isp;            /* s */
    double g0;             /* 9.81 (CRTBP_prop_EP_deriv.jl:41) */
    double default_mass;   /* 1000 kg when nstate == 6 (CRTBP_prop_EP_deriv.jl:20) */
    double tol;            /* LTO_ADAPTIVE only */
    int32_t mode;          /* LTO_FIXED | LTO_ADAPTIVE */
    int32_t err_norm;      /* LTO_ADAPTIVE only: LTO_NORM_* */
    int32_t max_attempts;  /* LTO_ADAPTIVE only; 0 -> 100000 */
    int32_t kernel;        /* LTO_KERNEL_* */
} lto_direct_params;

/* The params tuple of the indirect solver (multiShoot_CRTBP_indirect.jl:260) + tolerances (:79). */
typedef struct lto_indirect_params {
    double MU, DU, TU;
    double thrustLimit;    /* N */
    double mass;           /* kg (ndim == 12: constant mass) */
    double time_direction; /* +1 / -1 */
    double p, rho;         /* control law (CRTBP_stateCostate_deriv.jl:36-53) */
    double Isp, g0;        /* ndim == 14 only */
    double reltol, abstol; /* 1e-13 in the reference */
    int32_t controller;    /* LTO_CTRL_* */
    int32_t err_norm;      /* LTO_NORM_*; jac calls default to STATE_SENS (ForwardDiff semantics) */
    int32_t max_attempts;  /* 0 -> 100000 */
    int32_t kernel;        /* LTO_KERNEL_* */
} lto_indirect_params;

void lto_direct_params_default(lto_direct_params* p);      /* Earth-Moon constants, Isp 2000, FIXED */
void lto_indirect_params_default(lto_indirect_params* p);  /* Earth-Moon constants, 1e-13, p=1, rho=1 */

/* ---- lifetime ---------------------------------------------------------- */
int lto_version(void);
int lto_device_count(void);
int lto_init(int device, lto_handle** h);      /* LTO_ERR_NODEVICE when no sm_100 GPU */
/* One handle over several GPUs of the box, for a single host process (the Julia drop-in): every
 * host-buffer entry point splits its segments (trajectory forms: whole trajectories) into equal
 * contiguous ranges, one per device, runs them concurrently (one worker thread per device) and
 * each device copies its slab of the outputs into the caller's arrays (lto_indirect_newton and lto_indirect_solve_batch
 * included: whole trajectories per device, independent solver instances).  The device-pointer entry
 * points (lto_*_dev, lto_stream) need a single-device handle. */
int lto_init_devices(int n_devices, const int* devices, lto_handle** h);
int lto_n_devices(const lto_handle* h);
void lto_destroy(lto_handle* h);
const char* lto_last_error(const lto_handle* h);
void* lto_host_alloc(size_t bytes);            /* pinned host memory (NULL on failure) */
void lto_host_free(void* p);
/* counters since init / last reset: kernels launched, device ms of the last call's kernels */
int64_t lto_kernel_launches(const lto_handle* h);
double lto_last_kernel_ms(const lto_handle* h);
void* lto_stream(lto_handle* h);               /* cudaStream_t the *_dev entry points launch on */
/* Introspection (no device work): the chunk schedule the host-buffer entry points would use for their
 * H2D -> kernel -> D2H pipeline on a GPU with n_sm SMs.  method 0 = direct (nvar = nstate, nsteps and mode as in
 * lto_direct_*), 1 = indirect (nvar = ndim; nsteps and mode ignored); n_nodes = 0 pairs form, > 0 trajectory form (chunks are
 * whole trajectories).  Writes up to cap chunk sizes (segments) to chunks and returns the number of chunks, < 0 on bad arguments. */
int lto_host_chunk_plan(int method, int n_sm, int64_t n_seg, int n_nodes, int nvar, int nsteps, int mode, int want_jac,
                        int64_t* chunks, int cap);

/* ---- direct method, host buffers ---------------------------------------
 * pairs form: segment s goes from node a (Xa + s*nstate, ua + s*3, ta[s]) to node b.
 *   defect   nstate x n_seg            defect1[:, s]     (:101)
 *   errors   n_seg                     errors[s]         (:104)   (FIXED; 0 in ADAPTIVE)
 *   status   n_seg  (may be NULL)
 *   jac      per segment nstate x 2(nstate+3) column-major, column order
 *            [X_a, X_b, u_a, u_b] = rows (s-1)n+1..sn of Jac_temp (:125,:139-140)
 */
int lto_direct_defect(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int nstate, int nsteps,
                      const double* Xa, const double* Xb, const double* ua, const double* ub,
                      const double* ta, const double* tb,
                      double* defect, double* errors, int32_t* status);
int lto_direct_defect_jac(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int nstate, int nsteps,
                          const double* Xa, const double* Xb, const double* ua, const double* ub,
                          const double* ta, const double* tb,
                          double* defect, double* errors, int32_t* status, double* jac);
/* trajectory form: n_traj trajectories of n_nodes nodes each, stored back to back exactly
 * as the reference's X_all (nstate x n_nodes), u_all (3 x n_nodes), t_TU (n_nodes).
 * Segment (j, i) = trajectory j, nodes i -> i+1; outputs are indexed j*(n_nodes-1)+i. */
int lto_direct_defect_traj(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate,
                           int nsteps, const double* X_all, const double* u_all, const double* t_TU,
                           double* defect, double* errors, int32_t* status);
int lto_direct_defect_jac_traj(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate,
                               int nsteps, const double* X_all, const double* u_all, const double* t_TU,
                               double* defect, double* errors, int32_t* status, double* jac);

/* ---- indirect method, host buffers -------------------------------------
 *   x0        ndim x n_seg   (ndim = 12: [r v lr lv]; 14: [r v m lr lv lm])
 *   x_target  ndim x n_seg or NULL; defect = x(t1) - x_target (:82), x(t1) itself if NULL
 *   thrustLimit_seg, rho_seg: optional per-segment overrides of p->thrustLimit / p->rho
 *   status, nsteps_out (2 x n_seg: accepted, attempted) may be NULL
 *   phi       per segment ndim x ndim column-major = ForwardDiff.jacobian(f, x0) (:121)
 */
int lto_indirect_defect(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int ndim,
                        const double* x0, const double* t0, const double* t1, const double* x_target,
                        const double* thrustLimit_seg, const double* rho_seg,
                        double* defect, int32_t* status, int32_t* nsteps_out);
int lto_indirect_defect_jac(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int ndim,
                            const double* x0, const double* t0, const double* t1, const double* x_target,
                            const double* thrustLimit_seg, const double* rho_seg,
                            double* defect, int32_t* status, int32_t* nsteps_out, double* phi);
/* trajectory form: XC_all (ndim x n_nodes) per trajectory, t_TU (n_nodes) per trajectory;
 * thrustLimit_traj / rho_traj: optional per-TRAJECTORY overrides (continuation batches). */
int lto_indirect_defect_traj(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int ndim,
                             const double* XC_all, const double* t_TU,
                             const double* thrustLimit_traj, const double* rho_traj,
                             double* defect, int32_t* status, int32_t* nsteps_out);
int lto_indirect_defect_jac_traj(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int ndim,
                                 const double* XC_all, const double* t_TU,
                                 const double* thrustLimit_traj, const double* rho_traj,
                                 double* defect, int32_t* status, int32_t* nsteps_out, double* phi);

/* ---- device-resident variants ------------------------------------------
 * Same meaning, but every pointer is a DEVICE pointer on the handle's device and the
 * call only enqueues work on lto_stream(h) (no copies, no synchronisation).  n_nodes = 0
 * selects the pairs form (Xb/ub/tb used), n_nodes > 0 the trajectory form (Xb/ub/tb
 * ignored; n_seg = n_traj*(n_nodes-1)).  Optional outputs may be NULL; jac/phi NULL
 * selects the defect-only kernels. */
int lto_direct_dev(lto_handle* h, const lto_direct_params* p, int64_t n_seg, int n_nodes, int nstate, int nsteps,
                   const double* Xa, const double* Xb, const double* ua, const double* ub,
                   const double* ta, const double* tb,
                   double* defect, double* errors, int32_t* status, double* jac);
int lto_indirect_dev(lto_handle* h, const lto_indirect_params* p, int64_t n_seg, int n_nodes, int ndim,
                     const double* x0, const double* t0, const double* t1, const double* x_target,
                     const double* thrustLimit_arr, const double* rho_arr,
                     double* defect, int32_t* status, int32_t* nsteps_out, double* phi);
int lto_sync(lto_handle* h);   /* cudaStreamSynchronize(lto_stream(h)) */
/* out[r] = sum_i v[r*row_len + i]^2 on the device (enqueue-only, lto_stream): the merit value of the reference's
 * line searches, er[ind] = sum(defect[:].^2) (multiShoot_CRTBP_indirect.jl:241; multiShoot_CRTBP_direct.jl:425), one row
 * per trial trajectory, so that a batched line search returns one double per trial instead of every defect. */
int lto_sumsq_dev(lto_handle* h, const double* v, int64_t n_rows, int64_t row_len, double* out);

/* ---- Newton update and batched solver of the indirect method (device-side; SURVEY 8(f)) --------------
 * lto_indirect_newton: optimizeTraj_OLS's linear solve, src/multiShoot_CRTBP_indirect.jl:149-183,
 *     xc_update = -sparse(Jac_full) \ defect_vec
 * for n_traj trajectories of n_nodes nodes (12-dim: the reference's solver hard-codes the 12-dim RHS, :258), directly from
 * the Phi_i blocks and defects of lto_indirect_defect_jac_traj -- Jac_full (:127-142) is never formed.  The emptied columns
 * (first / last node's states :141-142; with flag_adjointsOnly every node's states :169-178) get a zero update, as
 * SuiteSparseQR's basic solution does.
 *   phi        per segment 12 x 12 column-major (n_traj*(n_nodes-1) blocks), 16-byte aligned
 *   defect     12 x (n_nodes-1) per trajectory
 *   xc_update  12 x n_nodes per trajectory (what optimizeTraj_OLS reshapes at :185)
 *   status     n_traj, LTO_ST_OK / LTO_ST_NAN (singular or non-finite system); may be NULL
 * The _dev form takes device pointers and only enqueues on lto_stream(h). */
int lto_indirect_newton(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                        const double* phi, const double* defect, double* xc_update, int32_t* status);
int lto_indirect_newton_dev(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                            const double* phi, const double* defect, double* xc_update, int32_t* status);
/* The second solve of optimizeTraj_OLS -- the second-order correction xc_update_soc = -Jac_sparse \ defect_vec with the SAME Jac_sparse
 * (:207) -- without factorising again: the handle keeps the factorisation of the last lto_indirect_newton_dev call (same n_traj,
 * n_nodes, flag_adjointsOnly required) and this call only transforms the new defects and back-substitutes.  `defect` 16-byte aligned. */
int lto_indirect_newton_resolve_dev(lto_handle* h, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                                    const double* defect, double* xc_update, int32_t* status);
/* lto_indirect_solve_batch: multiShoot_CRTBP_indirect (src/multiShoot_CRTBP_indirect.jl:58-345) for n_traj independent
 * trajectories at once, all arrays resident on the device between iterations: first nominal run (:274), then per
 * iteration jacobianCalc (:290), optimizeTraj_OLS with the second-order correction (:149-218; applied per trajectory where
 * norm(xc_update, Inf) < 1e-1), the 20-point line search from the 4th iteration on (:298-302, :221-246; all
 * 20 x n_traj trial trajectories in one launch), the update (:304) and the defect check (:328-336).  A trajectory stops
 * iterating exactly when the reference's loop would (er <= 1e-10, er > 1e3, NaN, or max_iter reached); the others go on.
 *   XC_all       in/out, 12 x n_nodes per trajectory (host)
 *   t_TU         n_nodes per trajectory
 *   thrustLimit_traj, rho_traj: optional per-trajectory overrides of p->thrustLimit / p->rho (continuation ladders)
 *   defect       out, 12 x (n_nodes-1) per trajectory, at the returned XC_all; may be NULL
 *   status_flag  out, n_traj: 0 converged, 1 max_iter / abort, 2 NaN (:282-286, :333-341); may be NULL
 *   iters        out, n_traj: iterations performed; may be NULL.   er_out: out, n_traj: final norm(defect, Inf); may be NULL */
int lto_indirect_solve_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes, int max_iter,
                             int flag_adjointsOnly, double* XC_all, const double* t_TU,
                             const double* thrustLimit_traj, const double* rho_traj,
                             double* defect, int32_t* status_flag, int32_t* iters, double* er_out);

/* The same four entry points for either system, ndim = 12 or 14 (anything else: LTO_ERR_ARG).  Every "12" above becomes ndim:
 * phi ndim x ndim column-major per segment, defect ndim x (n_nodes-1), xc_update / XC_all ndim x n_nodes per trajectory.  The
 * functions above are these with ndim = 12.
 *   ndim = 12  [r v | lr lv]: the end pins of :141-142 / :324-325 -- r, v (components 0..5) of the first and of the last node.
 *   ndim = 14  [r v m | lr lv lm] (the 14-dim system of lto_indirect_dev, p->Isp / p->g0 in the mass flow):
 *              first node r, v, m (components 0..6); last node r, v, lm (components 0..5 and 13).  The final mass is free and is
 *              solved for; lm, which enters no right-hand side, is held by its end value (otherwise the band is rank deficient).
 *              flag_adjointsOnly: the unknowns are the costates (7..13) of nodes 0..n_nodes-2 and m, lr, lv (6..12) of the last node.
 * Pinned components get exact-zero updates, so the batched solver leaves them bit-identical to the input ("the end states cannot
 * have moved").  A resolve must match the factorisation the handle holds in shape, mode AND ndim, or it is refused (LTO_ERR_ARG). */
int lto_indirect_newton_nd(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                           const double* phi, const double* defect, double* xc_update, int32_t* status);
int lto_indirect_newton_nd_dev(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                               const double* phi, const double* defect, double* xc_update, int32_t* status);
int lto_indirect_newton_resolve_nd_dev(lto_handle* h, int ndim, int64_t n_traj, int n_nodes, int flag_adjointsOnly,
                                       const double* defect, double* xc_update, int32_t* status);
int lto_indirect_solve_batch_nd(lto_handle* h, const lto_indirect_params* p, int ndim, int64_t n_traj, int n_nodes, int max_iter,
                                int flag_adjointsOnly, double* XC_all, const double* t_TU,
                                const double* thrustLimit_traj, const double* rho_traj,
                                double* defect, int32_t* status_flag, int32_t* iters, double* er_out);

/* lto_indirect_reduce_fuel_batch: the rho continuation of reduceFuel_indirect (src/HelperFunctions.jl:105-193) for n_traj independent
 * ladders in one call, every solver call on the device.  Each call is lto_indirect_solve_batch_nd's (maxIter = max_iter per call --
 * the reference uses 10 --, p = 1, flag_adjointsOnly = 0, per-trajectory rho and thrustLimit); the ladder logic runs on the device
 * between calls, and a ladder's next call starts as soon as its last one ended (not once per round):
 *   target = min(rho_target, rho_current); first call at rho_current from the start, done if it converges and rho_current == target;
 *   while calls fail and rho < 1: rho = min(5 rho, 1), from the start again (a failure at rho = 1 ends the ladder with that call);
 *   then, up to 100 rungs: after a success accept XC_new as the start and rho = max(rho / 2, target); after a failure
 *   rho *= 3 (1 + u) with u the trajectory's next back-off draw (:182); done on a success at rho <= target.
 *   ndim          12 or 14 (the 14-dim system with the pins and p->Isp described above)
 *   XC_all        in/out, ndim x n_nodes per trajectory: the starts on entry, the last call's XC_new on return
 *   t_TU          n_nodes per trajectory;  thrustLimit_traj: optional per-trajectory override of p->thrustLimit
 *   rho_current, rho_target: n_traj each;  backoff_uniform: n_traj x 100 doubles in [0, 1), consumed in order (at most 100 a ladder)
 *   defect        out, ndim x (n_nodes-1) per trajectory at the returned XC_all
 *   status        out, n_traj: the last call's status_flag (0, 1, 2), or 3 when the ladder gave up after 100 rungs
 *   calls, newton_iters, rho_last: out, n_traj: solver calls, Newton iterations over all calls, rho of the last call; may be NULL
 * p->p must be 1 (rho only means something there): anything else is LTO_ERR_ARG. */
int lto_indirect_reduce_fuel_batch(lto_handle* h, const lto_indirect_params* p, int ndim, int64_t n_traj, int n_nodes, int max_iter,
                                   double* XC_all, const double* t_TU, const double* thrustLimit_traj,
                                   const double* rho_current, const double* rho_target, const double* backoff_uniform,
                                   double* defect, int32_t* status, int32_t* calls, int32_t* newton_iters, double* rho_last);

/* ---- the linear subproblem of the direct solver (device-side; SURVEY 8(f) row 4) ------------------------
 * lto_direct_qp: optimizeTraj of src/multiShoot_CRTBP_direct.jl:248-403 in the setting the demo runs (flagEnd = false,
 * allowImpulsive = false): with tf_jump, p1_jump, p2_jump and the dV jumps pinned by their bounds (:288-302) the JuMP / Ipopt model is
 * the equality-constrained convex QP   min sum_i w_i |u_i + du_i|^2  (:323-325, :367-368)   s.t.  defect + Jac_full [dX; du] = 0 (:337),
 * dX_1[1:6] = b0, dX_N[1:6] = bf (:374-375), dX_1[7] = b0[7] when nstate = 7 (:270) -- solved exactly through its banded KKT system,
 * one warp per trajectory, straight from the Jacobian blocks of lto_direct_defect_jac[_traj] (Jac_full is never assembled).
 *   jac      per segment nstate x 2(nstate+3) column-major blocks, as lto_direct_defect_jac_traj returns them
 *   defect   nstate x (n_nodes-1) per trajectory;  u_all 3 x n_nodes;  t_TU n_nodes (node weights w)
 *   b0       per trajectory 6 (nstate 6) or 7 (nstate 7) doubles: state_0 - X_all[1:6,1] - [0,0,0,dV1] (:374) [, mass - X_all[7,1]]
 *   bf       per trajectory 6 doubles: state_f - X_all[1:6,end] - [0,0,0,dV2] (:375)
 *   x_update nstate x n_nodes, u_update 3 x n_nodes per trajectory (X_jump, u_jump :391-392);  status n_traj (LTO_ST_NAN: singular), may be NULL */
int lto_direct_qp(lto_handle* h, int64_t n_traj, int n_nodes, int nstate, const double* jac, const double* defect,
                  const double* u_all, const double* t_TU, const double* b0, const double* bf,
                  double* x_update, double* u_update, int32_t* status);
int lto_direct_qp_dev(lto_handle* h, int64_t n_traj, int n_nodes, int nstate, const double* jac, const double* defect,
                      const double* u_all, const double* t_TU, const double* b0, const double* bf,
                      double* x_update, double* u_update, int32_t* status);

/* lto_direct_solve_batch: the SQP loop of multiShoot_CRTBP_direct (src/multiShoot_CRTBP_direct.jl:465-594) for n_traj independent
 * trajectories, resident on the device, in the demo's setting (flagEnd = false, allowImpulsive = false, dV1 = dV2 = 0, FIXED grid): first
 * nominal run (:486); per iteration jacobianCalc as one launch (:500), the QP of optimizeTraj (lto_direct_qp_dev), the 10-point line search
 * from iteration 11 on (:559-561, :405-430; all 10 x n_traj trials in one launch), the update (:563-564) and the defect check (:585-588).
 * As in the reference every trajectory does at least one iteration (er starts at 1.0, :490) and stops when its max defect <= 1e-6 (:491) or
 * after max_iter iterations; tau1, tau2 and tf do not move in this setting, so the end states are constants of the call.
 *   X_all (nstate x n_nodes), u_all (3 x n_nodes): in/out per trajectory;  t_TU: n_nodes per trajectory
 *   state_0, state_f: 6 doubles per trajectory = interpEndStates(tau1, tau2, ...) (:483);  mass: mass0 of :270 (nstate 7)
 *   defect: out, nstate x (n_nodes-1) per trajectory (may be NULL); iters, er_out: out, n_traj (may be NULL) */
int lto_direct_solve_batch(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nstate, int nsteps, int max_iter,
                           double* X_all, double* u_all, const double* t_TU, const double* state_0, const double* state_f, double mass,
                           double* defect, int32_t* iters, double* er_out);

/* lto_direct_costates_batch: the costates of n_traj nstate-6 direct solutions (the layout of lto_direct_solve_batch), from the dual
 * solution of optimizeTraj's QP at the given point.  One K1 launch for the Jacobian blocks at (X_all, u_all), one launch of K7's dual
 * instantiation: the multipliers lambda_i of segment i's defect rows, mapped to node costates with Jx(i, k) = the 6 x 6 block of segment i's
 * Jacobian in node k's columns,
 *     p_i = Jx(i, i)^T lambda_i (i < n_nodes-1),  p_{n_nodes-1} = -Jx(n_nodes-2, n_nodes-1)^T lambda_{n_nodes-2},
 *     [lr; lv](t_i) = -p_i / kappa^2,  kappa = default_mass / kthr = default_mass DU 1e3 / TU^2 (u in N = kappa x nondimensional acceleration).
 * At a KKT point of the energy-optimal direct problem these are the discrete costates of the 12-dim p = 2 system (whose law a = -lv / 2
 * then gives lv(t_i) ~ -2 u_i / kappa), a start for lto_indirect_solve_batch at a thrust limit that does not bind.  The X_i rows of the KKT
 * system carry no objective term, so both one-sided values of an interior node agree up to the band solve's rounding.  nstate 7 is not
 * accepted (the X layout is 6 x n_nodes): the direct nstate-7 objective is not the 14-dim law's cost, so lm has no such map.
 *   X_all 6 x n_nodes, u_all 3 x n_nodes, t_TU n_nodes (finite, strictly increasing), state_0 / state_f 6: per trajectory
 *   XC_all       out, 12 x n_nodes per trajectory: rows 0-5 X_all bitwise, rows 6-11 the costates (NaN where status != LTO_ST_OK)
 *   multipliers  out, 6 x (n_nodes-1) per trajectory, lambda_i as solved; may be NULL
 *   du_max       out, n_traj: max |du| in N of the QP's control step at the given point (0 at an exact KKT point); may be NULL
 *   status       out, n_traj: the worst of the K1 segment statuses and K7's singular flag (LTO_ST_*); may be NULL
 * p->mode must be LTO_FIXED.  Null arrays, n_nodes < 2, non-finite t_TU / state_0 / state_f and a t_TU that is not strictly increasing are
 * LTO_ERR_ARG, naming the first offending trajectory; non-finite X_all / u_all show up in that trajectory's status.  n_traj = 0 does
 * nothing.  Inputs go up in one copy and the call synchronises once.  Multi-device handles split whole trajectories. */
int lto_direct_costates_batch(lto_handle* h, const lto_direct_params* p, int64_t n_traj, int n_nodes, int nsteps,
                              const double* X_all, const double* u_all, const double* t_TU,
                              const double* state_0, const double* state_f,
                              double* XC_all, double* multipliers, double* du_max, int32_t* status);

/* lto_stack_guess_batch: the demos' trajectory-stacking initial guess (CRTBP_Multishoot_direct_demo.jl:117-157, with interpInitialStates /
 * find_τ of src/HelperFunctions.jl:18-48) for n_traj transfers in one call, every stage on the device.  Per trajectory j:
 *   state_0 = spline(X0)(tau1[j]);  arc 1 = [state_0; 0] propagated from t_TU[0] to every node with t_TU < t_split (strict) and to t_split;
 *   tau2_0 = find_τ(Xf, arc-1 end);  arc 2 = [spline(Xf)(tau2_0); 0] from t_split to every remaining node and to t_TU[end];
 *   tau2 = find_τ(Xf, arc-2 end);  state_f = spline(Xf)(tau2);  XC_all = the arcs at the nodes, node 0 [state_0; 0], the last [state_f; 0].
 * spline(X): a natural cubic spline per row of the 6 x n table on LinRange(0, 1, n) (n >= 3), tau wrapped by +-1 steps into [0, 1];
 * find_τ: the first of tau = 0, 0.001, ..., 1 whose spline state is nearest (Euclidean) to the given state.  The arcs integrate the
 * 12-dim system with p as given and no STM (zero costates: the control is zero, the arcs are ballistic for any thrustLimit).
 *   X0_states, Xf_states  6 x n0, 6 x nf column-major orbit tables (finite)
 *   tau1, t_split         n_traj each: |tau1| <= 1e3, t_TU[0] < t_split <= t_TU[end]
 *   t_TU                  n_nodes per trajectory, finite and strictly increasing (n_nodes >= 2)
 *   XC_all                out, 12 x n_nodes per trajectory;  tau2: out, n_traj;  state_0, state_f: out, 6 per trajectory
 *   status                out, n_traj (may be NULL): the worst LTO_ST_* (largest code) of the trajectory's arc segments
 * A bad argument is LTO_ERR_ARG naming the first offending trajectory.  Multi-device handles split whole trajectories. */
int lto_stack_guess_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes,
                          const double* X0_states, int n0, const double* Xf_states, int nf,
                          const double* tau1, const double* t_TU, const double* t_split,
                          double* XC_all, double* tau2, double* state_0, double* state_f, int32_t* status);

/* lto_indirect_cost_batch: the control cost of n_traj 12-dim indirect trajectories (trajectory form, as lto_indirect_defect_traj) in one
 * call.  Every segment is integrated by the defect-only kernel K4 with two quadratures riding on its accepted steps, with the weights b
 * of the 8th-order update: int |a_u| dt and int |a_u|^2 dt, |a_u| = the control law's thrust-acceleration magnitude
 * (CRTBP_stateCostate_deriv.jl:36-53; 0 where |lv| = 0).  They are not in the error norm, so the steps and states are bitwise those of
 * lto_indirect_defect_traj; a trajectory's segments are summed in segment order, so its result does not depend on the batch around it.
 *   XC_all, t_TU, thrustLimit_traj, rho_traj: as lto_indirect_defect_traj with ndim = 12 (t_TU finite and non-decreasing)
 *   dv        out, n_traj: int |a_u| dt * DU 1e3 / TU, in m/s
 *   energy    out, n_traj: int (|a_u| mass DU 1e3 / TU^2)^2 dt, in N^2 TU (the units of the direct method's quadCost)
 *   defect    out, 12 x (n_nodes-1) per trajectory, the same output lto_indirect_defect_traj produces; may be NULL
 *   status    out, n_traj: the worst LTO_ST_* (largest code) of the trajectory's segments; may be NULL.  A trajectory with a segment
 *             whose status is not LTO_ST_OK has dv = energy = NaN (that segment never reached its end time)
 * The reference has no cost arithmetic to compare against: the quadrature is pinned by the constant-thrust closed form (p = 0) and an
 * independent DOP853 integration of the augmented 14-component system (tests/test_gpu_transfer_cost.py).
 * p->controller must be LTO_CTRL_RMS and p->kernel not LTO_KERNEL_GENERIC (the quadrature lives in K4): otherwise LTO_ERR_ARG, as for a
 * reversed or non-finite span (naming the first offending trajectory).  Multi-device handles split whole trajectories. */
int lto_indirect_cost_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes,
                            const double* XC_all, const double* t_TU,
                            const double* thrustLimit_traj, const double* rho_traj,
                            double* dv, double* energy, double* defect, int32_t* status);

/* lto_indirect_switch_batch: the switch times of n_traj 12-dim p = 1 indirect trajectories (trajectory form, as lto_indirect_defect_traj)
 * in one call.  Switching function S = |lv| - 1 (n = sqrt of the fma sum, as the kernels form it): thrust on where S > 0, off where
 * S <= 0.  Every segment is integrated by the defect-only kernel K4; on each accepted step [t, t + h] S is sampled at theta = k/8 on the
 * quintic Hermite interpolant of lv from both ends' (lv, h lv', h^2 lv'') (lv'' = U(r) lv - C^T lv', no extra right-hand sides) and each
 * sign change is refined by safeguarded Newton on that polynomial.  At an interior node, S on opposite sides at segment i's propagated end
 * and at node i + 1 is one switch at t_{i+1}, in the direction of node i + 1's side.  The scan is not in the error norm, so the steps and
 * defects are bitwise those of lto_indirect_defect_traj; a trajectory's segments are assembled in order, so its result does not depend on
 * the batch around it.
 *   XC_all, t_TU, thrustLimit_traj, rho_traj: as lto_indirect_defect_traj with ndim = 12 (t_TU finite and non-decreasing)
 *   max_switch  1 .. 64: switch slots per trajectory
 *   t_switch    out, max_switch per trajectory: the first max_switch switch times in TU, in time order (NaN in unused slots)
 *   direction   out, max_switch per trajectory: +1 a burn starts (off -> on), -1 a burn ends (0 in unused slots); they alternate, the
 *               first opposite to on_start
 *   n_switch    out, n_traj: the trajectory's true number of switches (it may exceed max_switch); -1 where status is not LTO_ST_OK
 *   on_start    out, n_traj: 1 where S > 0 at node 0
 *   defect      out, 12 x (n_nodes-1) per trajectory, the same output lto_indirect_defect_traj produces; may be NULL
 *   status      out, n_traj: the worst LTO_ST_* (largest code) of the trajectory's segments; may be NULL
 * p->p must be 1, p->controller LTO_CTRL_RMS and p->kernel not LTO_KERNEL_GENERIC (the scan lives in K4): otherwise LTO_ERR_ARG, as for
 * max_switch out of range or a reversed or non-finite span (naming the first offending trajectory).  Multi-device handles split whole
 * trajectories. */
int lto_indirect_switch_batch(lto_handle* h, const lto_indirect_params* p, int64_t n_traj, int n_nodes,
                              const double* XC_all, const double* t_TU,
                              const double* thrustLimit_traj, const double* rho_traj, int max_switch,
                              double* t_switch, int32_t* direction, int32_t* n_switch, int32_t* on_start,
                              double* defect, int32_t* status);

/* ---- peer memory: one process per GPU, results delivered to the solver rank without a collective --------
 * The rank that runs the Newton step allocates its full output arrays with lto_dev_alloc and exports them
 * (lto_ipc_export: a 64-byte cudaIpcMemHandle_t to send to the other processes by any means); every other rank
 * maps them (lto_ipc_open, NVLink peer access) and passes the mapped addresses, offset to its own slab, as the OUTPUT
 * pointers of lto_direct_dev / lto_indirect_dev: the kernels' epilogue stores then travel over NVLink into the solver
 * rank's HBM while the kernel is still computing (fused compute + gather, no SM taken from the propagation).
 * lto_push_async is the DMA-engine alternative: copy a finished local chunk to (peer) memory on the copy stream,
 * ordered after the work enqueued so far on lto_stream. */
void* lto_dev_alloc(lto_handle* h, size_t bytes);
void lto_dev_free(lto_handle* h, void* p);
int lto_ipc_export(lto_handle* h, void* dev_ptr, void* handle64);
int lto_ipc_open(lto_handle* h, const void* handle64, void** dev_ptr);
int lto_ipc_close(lto_handle* h, void* dev_ptr);
int lto_push_async(lto_handle* h, void* dst, const void* src, size_t bytes);
int lto_sync_copies(lto_handle* h);
/* Stream-ordered flags on lto_stream: lto_signal_dev writes `value` to the 64-bit word at `flag` (device or peer-mapped
 * memory) once everything enqueued before it has completed; lto_wait_dev holds the stream until *flag >= value. */
int lto_signal_dev(lto_handle* h, void* flag, uint64_t value);
int lto_wait_dev(lto_handle* h, void* flag, uint64_t value);

/* FP64 issue-rate probe used by bench.py for the roofline denominator: runs a
 * register-resident DFMA loop on every SM and returns achieved FLOP/s (FMA = 2). */
int lto_fp64_peak_probe(lto_handle* h, int iters, double* flops_per_s, double* ms);

/* Diagnostics: with LTO_ICW_PROF=1 in the environment at lto_init, the indirect throughput kernel
 * records per-warp cycle counters ([CTA][warp][work, wait, count, alive]); this copies them out. */
int lto_debug_profile(lto_handle* h, unsigned long long* out, int n_words);

#ifdef __cplusplus
}
#endif
#endif /* LTO_B200_H */
