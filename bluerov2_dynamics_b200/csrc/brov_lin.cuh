// brov_lin.cuh — exact Jacobians of the discrete step along batched trajectories (brov_linearize, include/brov.h):
// the arguments of linearize_kernel and its launcher (brov_lin.cu).
#pragma once
#include "brov_device.cuh"

namespace brov {

// Augmented state z = [x (NX) | Z (allocation-projected lag [6][3], thruster model only)], columns of J = [A | B]:
// NC = NZ + NU.  A block holds V = floor(128 / NC) vehicles, one thread per (vehicle, column).
template <int MODEL> struct LinDim {
    static constexpr int NX = ModelDim<MODEL>::NX;
    static constexpr int NU = ModelDim<MODEL>::NU;
    static constexpr int NZ = NX + (MODEL == MODEL_THRUSTER8 ? 18 : 0);
    static constexpr int NC = NZ + NU;
    static constexpr int V = 128 / NC;
    static constexpr int THREADS = V * NC;
};

struct LinArgs {
    Consts<double> c;             // engine constants (coefficients, allocation, lag discretisation of this dt)
    const double* z0;             // [n][NZ]
    const double* U;              // element (step k, vehicle i, channel j) at U[k*ust + i*usn + j]
    long long ust, usn;
    double* z_out;                // [n][NZ] or nullptr (may alias z0)
    double* z_traj;               // [steps][n][NZ] or nullptr
    double* jac;                  // [steps][n][NZ][NC]
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    long long n;
    int steps;
};

// fp64; thruster8, wrench12, quat13; RK4 / Euler
cudaError_t launch_linearize(int model, int integ, const LinArgs& a, cudaStream_t st);

}  // namespace brov
