// lto_ladder.h -- the rho-continuation ladder of reduceFuel_indirect (HelperFunctions.jl:105-193) as a per-trajectory state
// machine, compiled for the host (tests) and the device (lto_indirect_reduce_fuel_batch, lto_solve.cu).
//
// It is solvers._reduceFuel_steps branch for branch.  ladder_init() gives the rho of the first solver call (from the start);
// after every call, ladder_step() is given that call's status and either asks for another call (returns 1; `rho` is the call's
// rho, and `*accept` says whether the call's XC_new became the new start) or ends the ladder (returns 0; `*final_status` is the
// last call's status, or 3 when the ladder gave up after 100 rungs).  Every call starts from the last accepted XC_all.
// The back-off draws u in [0, 1) of `rho *= 3(1 + u)` (:182) come from the caller, at most LADDER_DRAWS of them, consumed in order.
#pragma once

#if defined(__CUDACC__)
#define LTO_LADDER_FN __host__ __device__ inline
#else
#define LTO_LADDER_FN inline
#endif

#define LADDER_DRAWS 100

struct LadderState {
    double rho, target;
    int phase;          // 0: the first call is out; 1: the x5 ramp (:131-141); 2: the main loop (:155-187)
    int count;          // main-loop rungs taken
    int draws;          // back-off draws consumed
};

LTO_LADDER_FN double ladder_init(LadderState* s, double rho_current, double rho_target) {
    s->target = rho_target > rho_current ? rho_current : rho_target;
    s->rho = rho_current;
    s->phase = 0; s->count = 0; s->draws = 0;
    return s->rho;
}

// Python's min(a, b) / max(a, b) return `a` unless `b` is strictly smaller / larger.
LTO_LADDER_FN int ladder_step(LadderState* s, int status, const double* draws, int* accept, int* final_status) {
    *accept = 0;
    if (s->phase == 0 && status == 0 && s->rho == s->target) { *final_status = status; return 0; }
    if (s->phase <= 1) {
        if (status != 0 && s->rho < 1) {                                       // while status != 0 and rho_temp < 1
            const double r5 = s->rho * 5;
            s->rho = 1.0 < r5 ? 1.0 : r5;
            s->phase = 1;
            return 1;
        }
        if (s->rho == 1 && status != 0) { *final_status = status; return 0; }
        if (status == 0) *accept = 1;
        s->phase = 2; s->count = 0;
    }
    if (!(s->rho > s->target || status != 0)) { *final_status = status; return 0; }
    s->count += 1;
    if (s->count > 100) { *accept = 0; *final_status = 3; return 0; }
    if (status == 0) {
        *accept = 1;
        const double h = s->rho / 2;
        s->rho = s->target > h ? s->target : h;
    } else {
        s->rho *= 3 * (1 + draws[s->draws++]);
    }
    return 1;
}
