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

// rows of ADJ_THREADS doubles in the dynamic shared memory of adjoint_coef_kernel: the RK4 stage buffer (3 NX), the
// coefficient cotangent (ADJ_NKPG) and, PV, the staged vehicle table (KP_COUNT)
__host__ __device__ constexpr int adjoint_coef_stage_rows(int model, int integ) {
    return integ == INTEG_RK4 ? 3 * (model == MODEL_QUAT13 ? 13 : 12) : 0;
}
constexpr size_t adjoint_coef_smem_bytes(int model, int integ, bool pv) {
    return (size_t)(adjoint_coef_stage_rows(model, integ) + ADJ_NKPG + (pv ? KP_COUNT : 0)) * ADJ_THREADS * sizeof(double);
}

// adjoint_kernel plus the coefficient cotangent (brov_rollout_vjp_coef): same models, integrators and a as launch_adjoint
cudaError_t launch_adjoint_coef(int model, int integ, const AdjCoefArgs& a, cudaStream_t st);

}  // namespace brov
