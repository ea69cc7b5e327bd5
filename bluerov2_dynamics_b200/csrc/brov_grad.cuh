// brov_grad.cuh — exact coefficient gradient and Gauss-Newton matrix of the sliding-window endpoint error
// (brov_multistep_se_grad, include/brov.h): the arguments of se_grad_kernel and its launcher (brov_grad.cu).
#pragma once
#include "brov_kernels.cuh"

namespace brov {

constexpr int GRAD_BLOCK = 128;
// Partials are written per block of a fixed grid that steps through the window tiles, so the workspace is
// GRAD_MAX_GRID x MAX_H x (1 + p + p(p+1)/2) doubles whatever the series length (23 MB at p = 36).
constexpr int GRAD_MAX_GRID = 1024;
constexpr int GRAD_DIR_PITCH = KP_COUNT + 1;   // odd pitch (in doubles) of the direction rows in shared memory

struct GradArgs {
    Consts<double> c;        // engine constants (allocation, lag discretisation, dt); c.kp is not read, c.has_current
                             // says whether the point or some direction has an ocean current
    const double* X;         // [rows][NX]
    const double* U;         // [rows][NU]
    const double* kp;        // [KP_COUNT] the point theta
    const double* dirs;      // [p][KP_COUNT] d kp / d theta_j
    const double* lag0;      // per-window initial lag or nullptr (zeros): [nwin][24] or, lag0_w, projected [nwin][18]
    int lag0_w;
    double* partial;         // [gridDim.x][MAX_H][ne]
    unsigned long long* health;   // [2] or nullptr; zeroed before the launch
    double eps;
    long long off;           // local row of window 0 (window0 - row0)
    int rows, nwin, nH;
    int H[MAX_H];            // ascending
    int p;                   // directions
    int W;                   // windows per tile: floor(GRAD_BLOCK / p)
    int ntiles;
    int ne;                  // accumulated entries per horizon: se, p gradient entries, p(p+1)/2 of the upper triangle
};

// launches se_grad_kernel (fp64; thruster8, wrench12, quat13; RK4 / Euler) on at most min(resident blocks,
// GRAD_MAX_GRID) blocks and the finish kernel: se_out [MAX_H], grad_out [MAX_H][p], gn_out [MAX_H][p][p]
cudaError_t launch_se_grad(int model, int integ, GradArgs& a, int num_sms, double* se_out, double* grad_out,
                           double* gn_out, cudaStream_t st);

}  // namespace brov
