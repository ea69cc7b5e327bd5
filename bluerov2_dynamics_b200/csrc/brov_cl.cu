// brov_cl.cu — closed-loop batched rollouts: an affine state-feedback law evaluated in the kernel at the start of every
// integrator step.
//
//   closed_loop_kernel   one thread per vehicle, the scheme of rollout_kernel: fp64 constants staged in shared memory,
//                        per-vehicle coefficients as ParamsShared (fp64) / ParamsRegs (fp32), the state and the
//                        allocation-projected lag in registers.  At step k the thread forms dz = z_k - zr_k from its
//                        registers (Euler angles wrapped to one turn), u_k = clamp(ur_k - K_k dz), optionally adds the
//                        stage cost, and takes integrate_step — the very step of the open-loop rollout — with u_k.
//
// Gains: a K shared by every vehicle and step is staged once per block in shared memory (<= 1.9 KB) and read as
// broadcasts; time-varying shared operands are read at the same address by every lane (one broadcast transaction per
// warp); per-vehicle operands are read directly.  Every product and sum of the feedback and of the cost is an explicit
// fma in a fixed order, so the result does not depend on where an operand lives: the four operand layouts give the
// same bits when they hold the same values.
#include "brov_cl.cuh"
#include "brov_kernels.cuh"

namespace brov {

__device__ __forceinline__ float rint_(float a) { return rintf(a); }
__device__ __forceinline__ double rint_(double a) { return rint(a); }
__device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }

// elements of the staged K, rounded up to 16 bytes (the snapshot tiles behind it are read as 128-bit vectors)
template <typename T, int NU, int NZ> struct KStage { static constexpr int N = (NU * NZ + 16 / (int)sizeof(T) - 1) / (16 / (int)sizeof(T)) * (16 / (int)sizeof(T)); };

template <typename T, int MODEL, int INTEG, bool PV, bool CU>
__global__ void __launch_bounds__(CL_MAX_BLOCK) __maxnreg__(MaxReg<T>::N)
closed_loop_kernel(const __grid_constant__ ClArgs<T> a) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    constexpr bool THR = MODEL == MODEL_THRUSTER8;
    constexpr int NL = THR ? 18 : 1;
    constexpr int NZ = NX + (THR ? 18 : 0);
    constexpr bool EULER_ANGLES = !ModelDim<MODEL>::QUAT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* smem = reinterpret_cast<T*>(smem_raw);

    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5;
    const long long gi = (long long)blockIdx.x * nthr + tid;
    const bool live = gi < a.n;
    const long long i = live ? gi : a.n - 1;   // dead lanes shadow the last vehicle, never store

    // fp64: the constant block in shared memory (as rollout_kernel, for the same reason)
    constexpr bool CSM = sizeof(T) == 8;
    __shared__ __align__(16) unsigned char cs_raw[CSM ? sizeof(Consts<T>) : 16];
    if constexpr (CSM) {
        const T* src = reinterpret_cast<const T*>(&a.c);
        T* dst = reinterpret_cast<T*>(cs_raw);
        for (int j = tid; j < (int)(sizeof(Consts<T>) / sizeof(T)); j += nthr) dst[j] = src[j];
    }
    const Consts<T>& cc = CSM ? *reinterpret_cast<const Consts<T>*>(cs_raw) : a.c;

    constexpr bool PVR = PvInRegs<T, PV>::V;
    typename std::conditional<PVR, ParamsRegs<T>,
                              typename std::conditional<PV, ParamsShared<T>, ParamsConst<T>>::type>::type p;
    if constexpr (PVR) {
#pragma unroll
        for (int j = 0; j < KP_COUNT; ++j) p.v[j] = __ldg(a.pv + (long long)j * a.n + i);
    } else if constexpr (PV) {
#pragma unroll 4
        for (int j = 0; j < KP_COUNT; ++j) smem[j * nthr + tid] = __ldg(a.pv + (long long)j * a.n + i);
        p.base = smem + tid;
        p.pitch = nthr;
        smem += KP_COUNT * nthr;
    } else {
        p.kp = cc.kp;
    }
    // the gains: staged once per block when one K serves every vehicle and step, else read where they are
    const T* Kp;
    if (a.k_smem) {
        for (int j = tid; j < NU * NZ; j += nthr) smem[j] = a.K[j];
        Kp = smem;
        smem += KStage<T, NU, NZ>::N;
    } else {
        Kp = a.K + i * a.K_sn;
    }
    __syncthreads();
    T* tile = smem + warp * 32 * NZ;   // per-warp snapshot tile [32][NZ] (NZ >= NU)

    T x[NX], lag[NL];
#pragma unroll
    for (int j = 0; j < NX; ++j) x[j] = a.z0[i * NZ + j];
#pragma unroll
    for (int j = 0; j < NL; ++j) lag[j] = THR ? a.z0[i * NZ + NX + j] : T(0);
    T cost = (a.cost && a.cost_accumulate) ? a.cost[i] : T(0);
    float mc = 1.0f;

    const T* zrp = a.zr + i * a.zr_sn;
    const T* urp = a.ur + i * a.ur_sn;
    const long long warp_v0 = (long long)blockIdx.x * nthr + warp * 32;
    const long long rem = a.n - warp_v0;
    const int warp_n = (int)(rem < 0 ? 0 : (rem > 32 ? 32 : rem));
    int countdown = a.stride;
    long long snap = 0;
    const T TWO_PI = T(6.283185307179586), INV_2PI = T(0.15915494309189535);
    NoSide side;

    for (int k = 0; k < a.steps; ++k) {
        const T* Kk = Kp + (long long)k * a.K_st;
        const T* zrk = zrp + (long long)k * a.zr_st;
        const T* urk = urp + (long long)k * a.ur_st;
        T u[NU];
#pragma unroll
        for (int r = 0; r < NU; ++r) u[r] = __ldg(urk + r);
        T s = T(0);
#pragma unroll
        for (int j = 0; j < NZ; ++j) {
            T d = (j < NX ? x[j] : lag[j < NX ? 0 : j - NX]) - __ldg(zrk + j);
            if (EULER_ANGLES && j >= 3 && j < 6) d = fma_(-TWO_PI, rint_(d * INV_2PI), d);
            s = fma_(a.q[j] * d, d, s);
#pragma unroll
            for (int r = 0; r < NU; ++r) u[r] = fma_(-Kk[r * NZ + j], d, u[r]);
        }
        // compare-select: a NaN input stays NaN (fmin / fmax would replace it by the bound)
#pragma unroll
        for (int r = 0; r < NU; ++r) u[r] = u[r] < a.u_min[r] ? a.u_min[r] : (u[r] > a.u_max[r] ? a.u_max[r] : u[r]);
        if (a.cost) {
#pragma unroll
            for (int r = 0; r < NU; ++r) {
                const T du = u[r] - __ldg(urk + r);
                s = fma_(a.r[r] * du, du, s);
            }
            cost += s;
        }
        // the input of a step that ends at a snapshot is stored before the step: u is not kept live across it
        if (countdown == 1 && a.u_traj)
            snapshot_warp<T, NU>(tile, u, a.u_traj + (snap * a.n + warp_v0) * NU, warp_n * NU, a.u_traj_vec != 0, lane);
        T acth;
        integrate_step<T, MODEL, INTEG, false, decltype(p), NoSide, CU>(cc, p, x, lag, u, acth, side);
        mc = fminf(mc, (float)acth);

        if (--countdown == 0) {
            countdown = a.stride;
            if (a.traj) {
                T z[NZ];
#pragma unroll
                for (int j = 0; j < NZ; ++j) z[j] = j < NX ? x[j] : lag[j < NX ? 0 : j - NX];
                snapshot_warp<T, NZ>(tile, z, a.traj + (snap * a.n + warp_v0) * NZ, warp_n * NZ, a.traj_vec != 0, lane);
            }
            ++snap;
        }
    }

    if (live) {
#pragma unroll
        for (int j = 0; j < NX; ++j) a.z_out[i * NZ + j] = x[j];
        if constexpr (THR) {
#pragma unroll
            for (int j = 0; j < NL; ++j) a.z_out[i * NZ + NX + j] = lag[j];
        }
        if (a.cost) a.cost[i] = cost;
    }
    if (a.health) {
        bool bad = false;
#pragma unroll
        for (int j = 0; j < NX; ++j) bad |= !finite_(x[j]);
        if constexpr (THR) {
#pragma unroll
            for (int j = 0; j < NL; ++j) bad |= !finite_(lag[j]);
        }
        count_health(Health{a.health, a.eps}, live && bad, live && ((double)mc < a.eps), lane);
    }
}

template <typename T, int MODEL, int INTEG, bool PV, bool CU>
static cudaError_t closed_loop_go(int block, const ClArgs<T>& a, cudaStream_t st) {
    constexpr int NZ = ModelDim<MODEL>::NX + (MODEL == MODEL_THRUSTER8 ? 18 : 0);
    constexpr int NU = ModelDim<MODEL>::NU;
    size_t smem = (a.traj || a.u_traj) ? (size_t)block * NZ * sizeof(T) : 0;
    if (a.k_smem) smem += (size_t)KStage<T, NU, NZ>::N * sizeof(T);
    if (PV && !PvInRegs<T, PV>::V) smem += (size_t)KP_COUNT * block * sizeof(T);
    auto kern = closed_loop_kernel<T, MODEL, INTEG, PV, CU>;
    if (smem > 16 * 1024) {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kern);
        if (e != cudaSuccess) return e;
        if (smem + fa.sharedSizeBytes > 48 * 1024) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
    }
    const long long grid = (a.n + block - 1) / block;
    kern<<<(unsigned)grid, block, smem, st>>>(a);
    return cudaGetLastError();
}

// CU = false: the build without the ocean-current terms (as the rollout's), chosen when no coefficient set has a current
template <typename T, int MODEL>
static cudaError_t closed_loop_model(int integ, int block, const ClArgs<T>& a, cudaStream_t st) {
    const bool pv = a.pv != nullptr, cur = a.c.has_current != 0;
    if (integ == INTEG_RK4) {
        if (pv) return cur ? closed_loop_go<T, MODEL, INTEG_RK4, true, true>(block, a, st)
                           : closed_loop_go<T, MODEL, INTEG_RK4, true, false>(block, a, st);
        return cur ? closed_loop_go<T, MODEL, INTEG_RK4, false, true>(block, a, st)
                   : closed_loop_go<T, MODEL, INTEG_RK4, false, false>(block, a, st);
    }
    if (pv) return cur ? closed_loop_go<T, MODEL, INTEG_EULER, true, true>(block, a, st)
                       : closed_loop_go<T, MODEL, INTEG_EULER, true, false>(block, a, st);
    return cur ? closed_loop_go<T, MODEL, INTEG_EULER, false, true>(block, a, st)
               : closed_loop_go<T, MODEL, INTEG_EULER, false, false>(block, a, st);
}

template <typename T> cudaError_t launch_closed_loop(int model, int integ, int block, const ClArgs<T>& a, cudaStream_t st) {
    if (a.n <= 0 || a.steps <= 0) return cudaSuccess;
    switch (model) {
        case MODEL_THRUSTER8: return closed_loop_model<T, MODEL_THRUSTER8>(integ, block, a, st);
        case MODEL_WRENCH12: return closed_loop_model<T, MODEL_WRENCH12>(integ, block, a, st);
        case MODEL_QUAT13: return closed_loop_model<T, MODEL_QUAT13>(integ, block, a, st);
    }
    return cudaErrorInvalidValue;
}

template cudaError_t launch_closed_loop<float>(int, int, int, const ClArgs<float>&, cudaStream_t);
template cudaError_t launch_closed_loop<double>(int, int, int, const ClArgs<double>&, cudaStream_t);

}  // namespace brov
