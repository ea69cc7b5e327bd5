// brov_cl.cuh — closed-loop batched rollouts with affine state feedback evaluated in the kernel (brov_closed_loop,
// include/brov.h): the arguments of closed_loop_kernel and its launcher (brov_cl.cu).
#pragma once
#include "brov_device.cuh"

namespace brov {

constexpr int CL_MAX_BLOCK = 128;
constexpr int CL_MAX_NZ = 30;

template <typename T> struct ClArgs {
    Consts<T> c;
    const T* z0;                  // [n][NZ]
    T* z_out;                     // [n][NZ] (may alias z0)
    // operand (step k, vehicle i, element e) at base[k*st + i*sn + e]; K rows are [NU][NZ]
    const T* K;
    long long K_st, K_sn;
    const T* zr;
    long long zr_st, zr_sn;
    const T* ur;
    long long ur_st, ur_sn;
    const T* pv;                  // per-vehicle coefficient table [KP_COUNT][n] or nullptr
    T* traj;                      // [steps / stride][n][NZ] or nullptr
    T* u_traj;                    // [steps / stride][n][NU] or nullptr
    T* cost;                      // [n] or nullptr
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    T u_min[8], u_max[8];
    T q[CL_MAX_NZ], r[8];
    long long n;
    int steps, stride;
    int cost_accumulate;
    int k_smem;                   // K is one matrix shared by every vehicle and step: staged in shared memory
    int traj_vec, u_traj_vec;     // 128-bit snapshot stores
};

// thruster8, wrench12, quat13; RK4 / Euler.  block: threads per block (32, 64 or 128)
template <typename T> cudaError_t launch_closed_loop(int model, int integ, int block, const ClArgs<T>& a, cudaStream_t st);

}  // namespace brov
