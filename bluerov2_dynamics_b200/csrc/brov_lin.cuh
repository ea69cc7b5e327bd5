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

// Extended Kalman filters (brov_ekf): one thread per (filter, state column), V = floor(128 / NX) filters per block.
// The covariance covers x only (NX x NX); the projected lag Z is a deterministic filter of the inputs.
template <int MODEL> struct EkfDim {
    static constexpr int NX = ModelDim<MODEL>::NX;
    static constexpr int NU = ModelDim<MODEL>::NU;
    static constexpr int NZ = LinDim<MODEL>::NZ;
    static constexpr int V = 128 / NX;
    static constexpr int THREADS = V * NX;
};

struct EkfArgs {
    Consts<double> c;
    const double* z0;             // [n][NZ]
    const double* P0;             // [n][NX][NX]
    // operand (step k, filter i, element j) at base[k*st + i*sn + j]; q and r at base[i*sn + j]
    const double* U;
    long long ust, usn;
    const double* Y;
    long long yst, ysn;
    const double* q;
    long long qsn;
    const double* r;
    long long rsn;
    double* z_out;                // [n][NZ] (may alias z0)
    double* P_out;                // [n][NX][NX] (may alias P0)
    double* x_traj;               // [steps / stride][n][NX] or nullptr
    double* P_traj;               // [steps / stride][n][NX][NX] or nullptr
    double* loglik;               // [n] or nullptr (the three together)
    double* nis;
    long long* count;
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    long long n;
    int steps, stride;
    int accumulate;
};

// fp64; thruster8, wrench12; RK4 / Euler
cudaError_t launch_ekf(int model, int integ, const EkfArgs& a, cudaStream_t st);

}  // namespace brov
