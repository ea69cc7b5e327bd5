// brov_grad.cu — forward-mode sensitivities of the sliding-window endpoint error in the kernel coefficients.
//
//   se_grad_kernel         one thread per (window, direction): the window's state as dual numbers along one direction
//                          of the coefficient vector, through the same RK4 / Euler step as integrate_step.  At every
//                          horizon the block gathers the endpoint tangents of its tile of windows in shared memory
//                          and adds the squared error, 2 r_w . t_j and the upper triangle of t_i . t_j into per-block
//                          accumulators; blocks step through the tiles of a fixed grid and write one partial each.
//   se_grad_finish_kernel  fixed-order sum of the partials (bit-reproducible, no floating-point atomics); both triangles
//                          of the Gauss-Newton matrix come from one sum, so it is exactly symmetric.
#include "brov_grad.cuh"

namespace brov {

// upper-triangle entry t (row-major over i <= j) -> (i, j)
__device__ __forceinline__ void tri_index(int t, int p, int& i, int& j) {
    i = 0;
    while (t >= p - i) { t -= p - i; ++i; }
    j = i + t;
}

template <int MODEL, int INTEG>
__global__ void __launch_bounds__(GRAD_BLOCK) se_grad_kernel(const __grid_constant__ GradArgs a) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    constexpr int NL = LagRegs<double, MODEL, false>::N;
    extern __shared__ double sm[];
    const int p = a.p, W = a.W, ne = a.ne, nH = a.nH;
    double* kps = sm;                               // [KP_COUNT]
    double* dks = kps + KP_COUNT;                   // [p][GRAD_DIR_PITCH]
    double* acc = dks + p * GRAD_DIR_PITCH;         // [nH][ne]
    double* tile = acc + nH * ne;                   // [W][p][NX] endpoint tangents
    double* res = tile + W * p * NX;                // [W][NX] endpoint residuals
    double* rss = res + W * NX;                     // [W] squared endpoint errors
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < KP_COUNT) kps[tid] = __ldg(a.kp + tid);
    for (int e = tid; e < p * KP_COUNT; e += GRAD_BLOCK) {
        const int j = e / KP_COUNT;
        dks[j * GRAD_DIR_PITCH + (e - j * KP_COUNT)] = __ldg(a.dirs + e);
    }
    for (int e = tid; e < nH * ne; e += GRAD_BLOCK) acc[e] = 0.0;
    __syncthreads();
    const int jd = tid % p, wl = tid / p;           // direction, window within the tile
    const bool live = wl < W;
    ParamsDual pd;
    pd.kp = kps;
    pd.dk = dks + (live ? jd : 0) * GRAD_DIR_PITCH;
    const int hmax = a.H[nH - 1];
    int n_bad = 0, n_sing = 0;
    for (int t = blockIdx.x; t < a.ntiles; t += gridDim.x) {
        const long long k0 = (long long)t * W;
        const long long k = k0 + wl;
        const bool act = live && k < a.nwin;
        const long long kr = k + a.off;
        // window k may run j steps while row k + j exists; the tile's first window has the most room
        const long long room0 = (long long)a.rows - 1 - (k0 + a.off);
        const int tsteps = (int)(room0 < hmax ? (room0 < 0 ? 0 : room0) : hmax);
        const long long room = (long long)a.rows - 1 - kr;
        const int nsteps = act ? (int)(room < hmax ? (room < 0 ? 0 : room) : hmax) : 0;
        Dual x[NX];
        double lag[NL];
#pragma unroll
        for (int q = 0; q < NX; ++q) x[q] = Dual(act ? __ldg(a.X + kr * NX + q) : 0.0);
        if (act) load_lag<double, MODEL, false>(a.c, a.lag0, a.lag0_w != 0, k, lag);
        else {
#pragma unroll
            for (int q = 0; q < NL; ++q) lag[q] = 0.0;
        }
        float mc = 1.0f;
        bool bad = false;
        for (int s = 0; s < tsteps; ++s) {
            const bool step = s < nsteps;           // windows at the end of the series stop early (masked)
            if (step) {
                double u[NU];
#pragma unroll
                for (int q = 0; q < NU; ++q) u[q] = __ldg(a.U + (kr + s) * NU + q);
                double acth;
                integrate_step_dual<MODEL, INTEG>(a.c, pd, x, lag, u, acth);
                mc = fminf(mc, (float)acth);
            }
#pragma unroll
            for (int h = 0; h < MAX_H; ++h) {
                if (h < nH && s + 1 == a.H[h]) {    // uniform over the block
                    if (live) {
#pragma unroll
                        for (int q = 0; q < NX; ++q) tile[(wl * p + jd) * NX + q] = step ? x[q].d : 0.0;
                        if (jd == 0) {
                            double ss = 0.0;
#pragma unroll
                            for (int q = 0; q < NX; ++q) {
                                const double e = step ? x[q].v - __ldg(a.X + (kr + s + 1) * NX + q) : 0.0;
                                res[wl * NX + q] = e;
                                ss += e * e;
                            }
                            rss[wl] = ss;
                            bad |= !(ss <= 1.7976931348623157e308);
                        }
                    }
                    __syncthreads();
                    double* ah = acc + h * ne;
                    for (int e = tid; e < ne; e += GRAD_BLOCK) {
                        double v = ah[e];
                        if (e == 0) {
                            for (int w = 0; w < W; ++w) v += rss[w];
                        } else if (e <= p) {
                            const int i = e - 1;
                            for (int w = 0; w < W; ++w) {
                                double d = 0.0;
#pragma unroll
                                for (int q = 0; q < NX; ++q) d = fma(res[w * NX + q], tile[(w * p + i) * NX + q], d);
                                v = fma(2.0, d, v);
                            }
                        } else {
                            int i, j;
                            tri_index(e - 1 - p, p, i, j);
                            for (int w = 0; w < W; ++w) {
                                double d = 0.0;
#pragma unroll
                                for (int q = 0; q < NX; ++q)
                                    d = fma(tile[(w * p + i) * NX + q], tile[(w * p + j) * NX + q], d);
                                v += d;
                            }
                        }
                        ah[e] = v;
                    }
                    __syncthreads();
                }
            }
        }
        if (act && jd == 0) {
            n_bad += bad ? 1 : 0;
            n_sing += ((double)mc < a.eps) ? 1 : 0;
        }
    }
    if (a.health) {
        const int tb = __reduce_add_sync(0xffffffffu, n_bad), ts = __reduce_add_sync(0xffffffffu, n_sing);
        if (lane == 0) {
            if (tb) atomicAdd(a.health + 0, (unsigned long long)tb);
            if (ts) atomicAdd(a.health + 1, (unsigned long long)ts);
        }
    }
    __syncthreads();
    double* out = a.partial + (long long)blockIdx.x * MAX_H * ne;
    for (int e = tid; e < nH * ne; e += GRAD_BLOCK) out[e] = acc[e];
}

// thread (h, e) sums the partials of every block in block order: same bits every run
static __global__ void __launch_bounds__(256) se_grad_finish_kernel(const double* __restrict__ partial, int nblocks,
                                                                    int nH, int p, int ne, double* __restrict__ se_out,
                                                                    double* __restrict__ grad_out,
                                                                    double* __restrict__ gn_out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= MAX_H * ne) return;
    const int h = idx / ne, e = idx - h * ne;
    double v = 0.0;
    if (h < nH)
        for (int b = 0; b < nblocks; ++b) v += partial[((long long)b * MAX_H + h) * ne + e];
    if (e == 0) {
        se_out[h] = v;
    } else if (e <= p) {
        grad_out[h * p + e - 1] = v;
    } else {
        int i, j;
        tri_index(e - 1 - p, p, i, j);
        gn_out[((long long)h * p + i) * p + j] = v;
        gn_out[((long long)h * p + j) * p + i] = v;
    }
}

static size_t grad_smem(const GradArgs& a, int nx) {
    return (size_t)(KP_COUNT + a.p * GRAD_DIR_PITCH + a.nH * a.ne + a.W * a.p * nx + a.W * nx + a.W) * sizeof(double);
}

template <int MODEL, int INTEG>
static cudaError_t se_grad_go(GradArgs& a, int num_sms, cudaStream_t st, int* grid_out) {
    auto kern = se_grad_kernel<MODEL, INTEG>;
    const size_t smem = grad_smem(a, ModelDim<MODEL>::NX);
    int nb = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, GRAD_BLOCK, smem);
    if (e != cudaSuccess) return e;
    long long grid = (long long)(nb > 0 ? nb : 1) * num_sms;
    if (grid > a.ntiles) grid = a.ntiles;
    if (grid > GRAD_MAX_GRID) grid = GRAD_MAX_GRID;
    kern<<<(unsigned)grid, GRAD_BLOCK, smem, st>>>(a);
    *grid_out = (int)grid;
    return cudaGetLastError();
}

template <int MODEL>
static cudaError_t se_grad_integ(int integ, GradArgs& a, int num_sms, cudaStream_t st, int* grid) {
    return integ == INTEG_RK4 ? se_grad_go<MODEL, INTEG_RK4>(a, num_sms, st, grid)
                              : se_grad_go<MODEL, INTEG_EULER>(a, num_sms, st, grid);
}

cudaError_t launch_se_grad(int model, int integ, GradArgs& a, int num_sms, double* se_out, double* grad_out,
                           double* gn_out, cudaStream_t st) {
    if (a.ntiles <= 0) return cudaErrorInvalidValue;
    int grid = 0;
    cudaError_t e = cudaErrorInvalidValue;
    switch (model) {
        case MODEL_THRUSTER8: e = se_grad_integ<MODEL_THRUSTER8>(integ, a, num_sms, st, &grid); break;
        case MODEL_WRENCH12: e = se_grad_integ<MODEL_WRENCH12>(integ, a, num_sms, st, &grid); break;
        case MODEL_QUAT13: e = se_grad_integ<MODEL_QUAT13>(integ, a, num_sms, st, &grid); break;
    }
    if (e != cudaSuccess) return e;
    const int n = MAX_H * a.ne;
    se_grad_finish_kernel<<<(n + 255) / 256, 256, 0, st>>>(a.partial, grid, a.nH, a.p, a.ne, se_out, grad_out, gn_out);
    return cudaGetLastError();
}

}  // namespace brov
