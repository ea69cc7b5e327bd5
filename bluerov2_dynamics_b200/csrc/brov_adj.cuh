// brov_adj.cuh — reverse-mode (adjoint) gradients of batched rollouts (brov_rollout_vjp, include/brov.h): the arguments
// of adjoint_kernel and its launcher (brov_adj.cu).
#pragma once
#include "brov_lin.cuh"

namespace brov {

// One thread per vehicle; the RK4 stage states of the step being reversed are staged in shared memory.
constexpr int ADJ_THREADS = 128;

struct AdjArgs {
    Consts<double> c;             // engine constants (coefficients, allocation, lag discretisation of this dt)
    const double* z0;             // [n][NZ]
    const double* U;              // element (step k, vehicle i, channel j) at U[k*ust + i*usn + j]
    long long ust, usn;
    const double* gtraj;          // [steps / stride][n][NX] or nullptr: cotangents of x at steps stride, 2 stride, ...
    const double* gzT;            // [n][NZ] or nullptr (zero)
    double* gz0;                  // [n][NZ] (may alias gzT)
    double* gU;                   // [steps][n][NU]
    double* z_out;                // [n][NZ] or nullptr
    double* ws;                   // [steps][NZ][n]: z_k of every step, vehicle index fastest
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    long long n;
    int steps, stride;
};

// bytes of the workspace of n vehicles over `steps` steps (NZ doubles per vehicle and step)
inline size_t adjoint_workspace_bytes(int nz, long long n, long long steps) {
    if (n <= 0 || steps <= 0) return 0;
    const unsigned long long per = (unsigned long long)nz * sizeof(double);
    if ((unsigned long long)n > ~0ULL / per / (unsigned long long)steps) return ~(size_t)0;
    return (size_t)((unsigned long long)n * (unsigned long long)steps * per);
}

// fp64; thruster8, wrench12, quat13; RK4 / Euler
cudaError_t launch_adjoint(int model, int integ, const AdjArgs& a, cudaStream_t st);

// coefficients with a gradient: KP_MINV .. KP_CUR + 2 (KP_ILAG1 and the pad entry are written as zero)
constexpr int ADJ_NKPG = KP_ILAG1;

struct AdjCoefArgs {
    AdjArgs a;
    double* gkp;                  // [KP_COUNT][n]: dL/dkp of each vehicle
    const double* pv;             // the per-vehicle table [KP_COUNT][n], or nullptr: the shared a.c.kp
};

// adjoint_kernel plus the coefficient cotangent (brov_rollout_vjp_coef): same models, integrators and a as launch_adjoint
cudaError_t launch_adjoint_coef(int model, int integ, const AdjCoefArgs& a, cudaStream_t st);

// Reverse-mode gradients of closed-loop rollouts (brov_closed_loop_vjp): the sweep closed_loop_adjoint_kernel and the
// fixed-order reductions of its per-(step, vehicle) operand cotangents into the operands' layouts.
struct ClAdjArgs {
    Consts<double> c;
    const double* z0;             // [n][NZ]
    // operand (step k, vehicle i, element e) at base[k*st + i*sn + e], as ClArgs; K rows are [NU][NZ]
    const double* K;
    long long K_st, K_sn;
    const double* zr;
    long long zr_st, zr_sn;
    const double* ur;
    long long ur_st, ur_sn;
    const double* pv;             // per-vehicle coefficient table [KP_COUNT][n] or nullptr
    const double* gtraj;          // [steps / stride][n][NZ] or nullptr
    const double* gzT;            // [n][NZ] or nullptr
    const double* gcost;          // [n] or nullptr (no cost term)
    double* gz0;                  // [n][NZ] (may alias gzT)
    double* z_out;                // [n][NZ] or nullptr
    double* ws;                   // [steps][NZ][n]: z_k, vehicle index fastest
    double* wgv;                  // [steps][NU][n] or nullptr: gv = dL/dv_k (v the unclamped feedback)
    double* wgur;                 // [steps][NU][n] or nullptr: dL/dur_k
    double* wgzr;                 // [steps][NZ][n] or nullptr: dL/dzr_k
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    double u_min[8], u_max[8];
    double q[30], r[8];
    long long n;
    int steps, stride;
    int k_smem;                   // K is one matrix shared by every vehicle and step: staged in shared memory
};

// bytes of n * (steps * per + scr) doubles: the workspace of brov_closed_loop_vjp with `per` doubles per vehicle and
// step (z_k and the requested operands' cotangents) and `scr` per vehicle (the scratch of a const_shared operand);
// SIZE_MAX when that does not fit in size_t
inline size_t cl_adjoint_bytes(unsigned long long per, unsigned long long scr, long long n, long long steps) {
    if (n <= 0 || steps <= 0) return 0;
    const unsigned long long un = (unsigned long long)n, ut = (unsigned long long)steps, lim = ~0ULL / sizeof(double);
    if (un > lim / per / ut) return ~(size_t)0;
    const unsigned long long a = un * ut * per;
    if (scr && un > (lim - a) / scr) return ~(size_t)0;
    return (size_t)((a + un * scr) * sizeof(double));
}
// every operand gradient requested: z, gv, gur, gzr per step, one [NU*NZ] scratch per vehicle
inline size_t cl_adjoint_workspace_bytes(int nz, int nu, long long n, long long steps) {
    return cl_adjoint_bytes((unsigned long long)(2 * nz + 2 * nu), (unsigned long long)nu * nz, n, steps);
}

// fp64; thruster8, wrench12, quat13; RK4 / Euler
cudaError_t launch_closed_loop_adjoint(int model, int integ, const ClAdjArgs& a, cudaStream_t st);

// One operand gradient out[k*st + i*sn + e] (the operand's own strides) from the sweep's cotangents:
//   which = 0: dL/dK  [NU][NZ] = -gv dz^T (dz recomputed from the stored z_k and zr)
//           1: dL/dzr [NZ] (wgzr)      2: dL/dur [NU] (wgur)
// Elements read by several (step, vehicle) pairs (a zero stride) receive the sum of their contributions, each in a
// fixed order; scratch: [NU*NZ][n] doubles, used when both strides are 0.
cudaError_t launch_closed_loop_adjoint_reduce(int model, int which, const ClAdjArgs& a, double* out, long long st,
                                              long long sn, double* scratch, cudaStream_t s);

}  // namespace brov
