// brov_kernels_impl.cuh — runtime -> template dispatch.  Included by brov_kernels_f32.cu / brov_kernels_f64.cu; each
// instantiates every (model, integrator, lag1, per-vehicle, generated-input) combination for its scalar type.
#pragma once
#include "brov_kernels.cuh"

namespace brov {

// dynamic shared memory of a rollout launch: [fp64 per-vehicle coefficient table][snapshot tiles]
template <typename T, int MODEL, bool PV> static size_t rollout_smem(bool traj) {
    constexpr int NX = ModelDim<MODEL>::NX;
    size_t smem = traj ? (size_t)ROLLOUT_BLOCK * NX * sizeof(T) : 0;
    if (PV && !PvInRegs<T, PV>::V) smem += (size_t)KP_COUNT * ROLLOUT_BLOCK * sizeof(T);
    return smem;
}

template <typename T, int MODEL, int INTEG, bool LAG1, bool PV, bool GEN, bool CU>
static cudaError_t rollout_launch(const RolloutArgs<T>& a, cudaStream_t st) {
    const int grid = ((a.n + ROLLOUT_BLOCK - 1) / ROLLOUT_BLOCK) * (a.quanta > 1 ? a.quanta : 1);
    const size_t smem = rollout_smem<T, MODEL, PV>(a.traj != nullptr);
    auto kern = rollout_kernel<T, MODEL, INTEG, LAG1, PV, GEN, CU>;
    if (smem > 16 * 1024) {
        // static + dynamic shared memory beyond 48 KB needs the opt-in (the fp64 coefficient table alone is 36 KB)
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kern);
        if (e != cudaSuccess) return e;
        if (smem + fa.sharedSizeBytes > 48 * 1024) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
    }
    kern<<<grid, ROLLOUT_BLOCK, smem, st>>>(a);
    return cudaGetLastError();
}

// resident blocks per SM of the kernel that launch_rollout would pick (for the temporal-tiling heuristic)
template <typename T, int MODEL, int INTEG, bool LAG1, bool PV, bool GEN, bool CU>
static int rollout_occ(bool traj) {
    int nb = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rollout_kernel<T, MODEL, INTEG, LAG1, PV, GEN, CU>,
                                                                  ROLLOUT_BLOCK, rollout_smem<T, MODEL, PV>(traj));
    return e == cudaSuccess ? nb : 0;
}

// runtime -> template dispatch; F is a generic lambda called with std::integral_constant tags
template <typename T, class F>
static auto rollout_dispatch(int model, int integ, bool lag1, bool pv, bool gen, bool cur, F&& f) {
    // CU tag: false = the common-case build of a streamed-input Fossen kernel (no ocean current, aligned per-vehicle
    // input rows: both decided at compile time), true = the general build (flags read at run time); `cur` = general
    auto with_flags = [&](auto M, auto L1) {
        auto with_integ = [&](auto I) {
            auto with_cur = [&](auto PV, auto G) {
                constexpr bool has_nocur = !decltype(G)::value && !ModelDim<decltype(M)::value>::DI;
                if constexpr (has_nocur) {
                    if (!cur) return f(M, I, L1, PV, G, std::false_type{});
                }
                return f(M, I, L1, PV, G, std::true_type{});
            };
            if (pv) return gen ? with_cur(std::true_type{}, std::true_type{}) : with_cur(std::true_type{}, std::false_type{});
            return gen ? with_cur(std::false_type{}, std::true_type{}) : with_cur(std::false_type{}, std::false_type{});
        };
        return integ == INTEG_RK4 ? with_integ(std::integral_constant<int, INTEG_RK4>{})
                                  : with_integ(std::integral_constant<int, INTEG_EULER>{});
    };
    using std::integral_constant;
    switch (model) {
        case MODEL_THRUSTER8: return with_flags(integral_constant<int, MODEL_THRUSTER8>{}, std::false_type{});
        case MODEL_WRENCH12:
            return lag1 ? with_flags(integral_constant<int, MODEL_WRENCH12>{}, std::true_type{})
                        : with_flags(integral_constant<int, MODEL_WRENCH12>{}, std::false_type{});
        case MODEL_QUAT13:
            return lag1 ? with_flags(integral_constant<int, MODEL_QUAT13>{}, std::true_type{})
                        : with_flags(integral_constant<int, MODEL_QUAT13>{}, std::false_type{});
        case MODEL_DI12_U8: return with_flags(integral_constant<int, MODEL_DI12_U8>{}, std::false_type{});
        case MODEL_DI12_U6: return with_flags(integral_constant<int, MODEL_DI12_U6>{}, std::false_type{});
        default: return with_flags(integral_constant<int, MODEL_DIQ13_U6>{}, std::false_type{});
    }
}

// the double-integrator models have no per-vehicle table (brov_set_vehicle_params refuses it): their PV kernels are
// never instantiated
template <int MODEL, bool PV> struct RolloutExists { static constexpr bool V = !(PV && ModelDim<MODEL>::DI); };

template <typename T>
int rollout_blocks_per_sm(int model, int integ, bool lag1, bool pv, bool gen, bool traj, bool cur) {
    if (model < MODEL_THRUSTER8 || model > MODEL_DIQ13_U6) return 0;
    return rollout_dispatch<T>(model, integ, lag1, pv, gen, cur, [&](auto M, auto I, auto L1, auto PV, auto G, auto CU) -> int {
        if constexpr (RolloutExists<decltype(M)::value, decltype(PV)::value>::V)
            return rollout_occ<T, decltype(M)::value, decltype(I)::value, decltype(L1)::value, decltype(PV)::value, decltype(G)::value,
                               decltype(CU)::value>(traj);
        else
            return 0;
    });
}

template <typename T>
cudaError_t launch_rollout(int model, int integ, bool lag1, const RolloutArgs<T>& a, cudaStream_t st) {
    if (a.n <= 0 || a.steps <= 0) return cudaSuccess;
    if (model < MODEL_THRUSTER8 || model > MODEL_DIQ13_U6) return cudaErrorInvalidValue;
    const bool general = a.c.has_current != 0 || !(a.u_vec && a.u_stride_n != 0);
    return rollout_dispatch<T>(model, integ, lag1, a.pv != nullptr, a.gen.on != 0, general,
                               [&](auto M, auto I, auto L1, auto PV, auto G, auto CU) -> cudaError_t {
        if constexpr (RolloutExists<decltype(M)::value, decltype(PV)::value>::V)
            return rollout_launch<T, decltype(M)::value, decltype(I)::value, decltype(L1)::value, decltype(PV)::value, decltype(G)::value,
                                  decltype(CU)::value>(a, st);
        else
            return cudaErrorInvalidValue;
    });
}

template <typename T> cudaError_t launch_lag_tail(const LagTailArgs<T>& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    if (a.gen.on) {
        lag_tail_gen_kernel<T><<<(a.n + RHS_BLOCK - 1) / RHS_BLOCK, RHS_BLOCK, 0, st>>>(a);
    } else {
        const long long threads = (long long)a.n * 8;
        lag_tail_kernel<T><<<(unsigned)((threads + TAIL_BLOCK - 1) / TAIL_BLOCK), TAIL_BLOCK, 0, st>>>(a);
    }
    return cudaGetLastError();
}

template <typename T> cudaError_t launch_gen_inputs(int nu, const GenInputsArgs<T>& a, cudaStream_t st) {
    if (a.n_sel <= 0 || a.steps <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((a.n_sel + RHS_BLOCK - 1) / RHS_BLOCK);
    if (nu == 8) gen_inputs_kernel<T, 8><<<grid, RHS_BLOCK, 0, st>>>(a);
    else gen_inputs_kernel<T, 6><<<grid, RHS_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

template <typename T, int MODEL, bool LAG1>
static cudaError_t rhs_go(const RhsArgs<T>& a, cudaStream_t st) {
    const int grid = (a.n + RHS_BLOCK - 1) / RHS_BLOCK;
    if (a.pv) {
        size_t smem = (size_t)KP_COUNT * RHS_BLOCK * sizeof(T);
        rhs_kernel<T, MODEL, LAG1, true><<<grid, RHS_BLOCK, smem, st>>>(a);
    } else {
        rhs_kernel<T, MODEL, LAG1, false><<<grid, RHS_BLOCK, 0, st>>>(a);
    }
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_rhs(int model, bool lag1, const RhsArgs<T>& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    switch (model) {
        case MODEL_THRUSTER8: return rhs_go<T, MODEL_THRUSTER8, false>(a, st);
        case MODEL_WRENCH12: return lag1 ? rhs_go<T, MODEL_WRENCH12, true>(a, st) : rhs_go<T, MODEL_WRENCH12, false>(a, st);
        case MODEL_QUAT13: return lag1 ? rhs_go<T, MODEL_QUAT13, true>(a, st) : rhs_go<T, MODEL_QUAT13, false>(a, st);
        case MODEL_DI12_U8: return rhs_go<T, MODEL_DI12_U8, false>(a, st);
        case MODEL_DI12_U6: return rhs_go<T, MODEL_DI12_U6, false>(a, st);
        case MODEL_DIQ13_U6: return rhs_go<T, MODEL_DIQ13_U6, false>(a, st);
    }
    return cudaErrorInvalidValue;
}

template <typename T> int se_blocks(long long nwin) {
    return (int)((nwin + ROLLOUT_BLOCK - 1) / ROLLOUT_BLOCK);
}

template <typename T, int MODEL>
static cudaError_t se_go(int integ, const SeArgs<T>& a, cudaStream_t st) {
    const int nblocks = se_blocks<T>((a.nwin + a.wpt - 1) / a.wpt) * (a.quanta > 1 ? a.quanta : 1);
    if (integ == INTEG_RK4) se_kernel<T, MODEL, INTEG_RK4><<<nblocks, ROLLOUT_BLOCK, 0, st>>>(a);
    else se_kernel<T, MODEL, INTEG_EULER><<<nblocks, ROLLOUT_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_se(int model, int integ, const SeArgs<T>& a, double* se_out, cudaStream_t st) {
    cudaError_t e = cudaErrorInvalidValue;
    switch (model) {
        case MODEL_THRUSTER8: e = se_go<T, MODEL_THRUSTER8>(integ, a, st); break;
        case MODEL_WRENCH12: e = se_go<T, MODEL_WRENCH12>(integ, a, st); break;
        case MODEL_QUAT13: e = se_go<T, MODEL_QUAT13>(integ, a, st); break;
        case MODEL_DI12_U8: e = se_go<T, MODEL_DI12_U8>(integ, a, st); break;
        case MODEL_DI12_U6: e = se_go<T, MODEL_DI12_U6>(integ, a, st); break;
        case MODEL_DIQ13_U6: e = se_go<T, MODEL_DIQ13_U6>(integ, a, st); break;
    }
    if (e != cudaSuccess) return e;
    se_finish_kernel<<<1, 256, 0, st>>>(a.partial, se_blocks<T>((a.nwin + a.wpt - 1) / a.wpt) * (a.quanta > 1 ? a.quanta : 1),
                                        se_out);
    return cudaGetLastError();
}

// the sweep serves the three Fossen models (the double integrator has no coefficient table to sweep)
template <typename T, int MODEL>
static cudaError_t se_sweep_go(int integ, const SweepArgs<T>& a, cudaStream_t st) {
    const unsigned grid = (unsigned)((long long)a.P * a.nwb);
    if (integ == INTEG_RK4) se_sweep_kernel<T, MODEL, INTEG_RK4><<<grid, ROLLOUT_BLOCK, 0, st>>>(a);
    else se_sweep_kernel<T, MODEL, INTEG_EULER><<<grid, ROLLOUT_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_se_sweep(int model, int integ, const SweepArgs<T>& a, double* se_out, cudaStream_t st) {
    if (a.P <= 0 || a.nwb <= 0) return cudaSuccess;
    cudaError_t e = cudaErrorInvalidValue;
    switch (model) {
        case MODEL_THRUSTER8: e = se_sweep_go<T, MODEL_THRUSTER8>(integ, a, st); break;
        case MODEL_WRENCH12: e = se_sweep_go<T, MODEL_WRENCH12>(integ, a, st); break;
        case MODEL_QUAT13: e = se_sweep_go<T, MODEL_QUAT13>(integ, a, st); break;
    }
    if (e != cudaSuccess) return e;
    se_sweep_finish_kernel<<<a.P, 256, 0, st>>>(a.partial, a.nwb, se_out);
    return cudaGetLastError();
}

template <typename T> cudaError_t launch_se_carry_lag(const CarryLagArgs<T>& a, cudaStream_t st) {
    if (a.nwin <= 0) return cudaSuccess;
    const long long threads = (a.nwin + a.wpt - 1) / a.wpt;
    se_carry_lag_kernel<T><<<(unsigned)((threads + RHS_BLOCK - 1) / RHS_BLOCK), RHS_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_reduced9(const Red9Consts<T>& c, const T* X, const T* U, T* O, long long B, cudaStream_t st) {
    if (B <= 0) return cudaSuccess;
    const long long grid = (B + RED9_BLOCK - 1) / RED9_BLOCK;
    const int vec = ((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(O)) & 15) == 0;
    reduced9_kernel<T><<<(unsigned)grid, RED9_BLOCK, 0, st>>>(c, X, U, O, B, vec);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_fma_peak(int iters, int blocks, T* scratch, cudaStream_t st) {
    fma_peak_kernel<T><<<blocks, 256, 0, st>>>(scratch, iters, T(0.999), T(1e-3));
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_thruster_wrench(const ThrusterArgs<T>& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    thruster_wrench_kernel<T><<<(a.n + RHS_BLOCK - 1) / RHS_BLOCK, RHS_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_thruster_series(const ThrusterSeriesArgs<T>& a, cudaStream_t st) {
    if (a.rows <= 0) return cudaSuccess;
    thruster_series_kernel<T><<<(unsigned)((a.rows + RHS_BLOCK - 1) / RHS_BLOCK), RHS_BLOCK, 0, st>>>(a);
    return cudaGetLastError();
}

#define BROV_INSTANTIATE(T)                                                                                         \
    template cudaError_t launch_rollout<T>(int, int, bool, const RolloutArgs<T>&, cudaStream_t);                   \
    template int rollout_blocks_per_sm<T>(int, int, bool, bool, bool, bool, bool);                                      \
    template cudaError_t launch_lag_tail<T>(const LagTailArgs<T>&, cudaStream_t);                                  \
    template cudaError_t launch_gen_inputs<T>(int, const GenInputsArgs<T>&, cudaStream_t);                         \
    template cudaError_t launch_rhs<T>(int, bool, const RhsArgs<T>&, cudaStream_t);                                \
    template cudaError_t launch_se<T>(int, int, const SeArgs<T>&, double*, cudaStream_t);                          \
    template int se_blocks<T>(long long);                                                                          \
    template cudaError_t launch_se_sweep<T>(int, int, const SweepArgs<T>&, double*, cudaStream_t);                 \
    template cudaError_t launch_se_carry_lag<T>(const CarryLagArgs<T>&, cudaStream_t);                             \
    template cudaError_t launch_reduced9<T>(const Red9Consts<T>&, const T*, const T*, T*, long long, cudaStream_t); \
    template cudaError_t launch_fma_peak<T>(int, int, T*, cudaStream_t);                                           \
    template cudaError_t launch_thruster_wrench<T>(const ThrusterArgs<T>&, cudaStream_t);                          \
    template cudaError_t launch_thruster_series<T>(const ThrusterSeriesArgs<T>&, cudaStream_t);

}  // namespace brov
