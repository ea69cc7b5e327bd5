// brov_kernels.cuh — the sm_100a kernels of the engine and their launchers (templated on the scalar type; the two
// translation units brov_kernels_f32.cu / brov_kernels_f64.cu instantiate them so nvcc can build them in parallel).
//
//   rollout_kernel   open-loop rollout of N vehicles, one thread per vehicle, optional strided trajectory
//                    writeback through per-warp shared-memory staging        (simulate_physics,
//                    training/train_tank_brov2_rk4.py:375-396 and its Euler twins)
//   rhs_kernel       one dynamics() call for N vehicles                       (fossen/BlueROV2.py:357-400 etc.)
//   se_kernel        sliding-window multi-horizon endpoint squared error, one thread per window, warp-shuffle +
//                    block reduction into per-block partial sums              (multistep_rmse_endpoint_physics,
//                    training/train_tank_brov2_rk4.py:399-417 and twins)
//   se_finish_kernel fixed-order sum of the per-block partials (bit-reproducible result)
//   reduced9_kernel  bluerov_compute RHS, shared-memory transposed, HBM-bound  (fossen/bluerov_torch.py:20-67)
//   fma_peak_kernel  FMA-chain microbenchmark: the FP32 / FP64 pipe roofline denominator measured in-run
#pragma once
#include <type_traits>
#include "brov_device.cuh"

namespace brov {

constexpr int MAX_H = 4;          // horizons per se launch
constexpr int RHS_BLOCK = 128;
constexpr int RED9_BLOCK = 256;
constexpr int TAIL_BLOCK = 256;
// Launch shape of the per-vehicle kernels — the fastest configuration measured on B200 (alternatives and their
// timings: profiles/r01e / r01g / r01i *.json, DESIGN.md section 4):
//   fp32: 128-thread blocks, 128-register cap (16 warps per SM), everything in registers;
//   fp64: 128-thread blocks, no register cap (~250 registers, 8 warps per SM), lag state and RK4 accumulator in
//         registers, next-step inputs prefetched, constant block in shared memory.
constexpr int ROLLOUT_BLOCK = 128;
// Register caps.  fp32: 128 (16 warps per SM) for every kernel, the Monte-Carlo ones included (per-vehicle
// coefficients in registers: 2.90 ms per 100 steps of 1,048,576 vehicles at 128, 2.99 at 168, 3.07 with the table in
// shared memory; profiles/r02d_tune_variants.txt).  fp64: none — the wrench-input kernels do fit 168 registers with
// the prefetch path, but 12 instead of 8 warps per SM bought 2 % (wrench12) / 6 % (quat13) and cost the Monte-Carlo
// kernel 30 % in spills (profiles/r02i_tune_variants.txt): they are bound by dependent-issue latency inside a stage,
// not by the number of warps.
// (fp32 Monte-Carlo kernel with 160 / 192 registers: 2.9995 / 2.9292 ms against 2.9848 ms at 128, r02t)
template <typename T> struct MaxReg { static constexpr int N = sizeof(T) == 8 ? 255 : 128; };
// Streamed inputs: every kernel prefetches the next step's command row into registers, requested between stages 2 and 3
// of the current step (LateSide, brov_device.cuh).  A per-warp TMA bulk-copy ring (cp.async.bulk + mbarrier, 4 steps
// ahead) was the input path of the lag-free fp64 and the fp32 Monte-Carlo kernels for most of round 2 — it beat a
// prefetch issued at the TOP of the step by 12-15 % there (r02g) — and was removed when the mid-step prefetch beat it
// in turn on every kernel (r02t batch 4, per launch: quat13 fp64 3.235 -> 3.034 ms, wrench12 fp64 3.281 -> 3.225 ms,
// Monte-Carlo fp64 0.442 -> 0.430 ms, Monte-Carlo fp32 2.987 -> 2.621 ms): the barrier wait at the top of the loop
// costs more than 16 registers held for half a step.
// where the per-vehicle coefficient table lives during a launch: fp32 registers, fp64 shared memory [36][BLOCK]
template <typename T, bool PV> struct PvInRegs { static constexpr bool V = PV && sizeof(T) == 4; };

// per-launch health accounting (optional): vehicles whose final state is not finite, vehicles that came within eps of
// the Euler-angle singularity theta = +-pi/2 (fossen/BlueROV2.py:43-62 clamps cos theta there)
struct Health {
    unsigned long long* counters;   // [2]: non-finite, near-singular; zeroed by the library before the launch
    double eps;
};

template <typename T> struct RolloutArgs {
    Consts<T> c;
    InputGen<T> gen;    // gen.on: inputs are generated in the kernel, U is ignored
    const T* x0;        // [n][NX]
    T* xT;              // [n][NX] (may alias x0)
    const T* U;         // element (k, i, j) at U[k*u_stride_t + i*u_stride_n + j]
    long long u_stride_t, u_stride_n;
    const T* lag_in;    // [n][NLAG] or nullptr (zeros); thruster model: 18 values if lag_in_w, else 24 (projected on load)
    T* lag_out;         // [n][NLAG] or nullptr; thruster model: allocation-projected [n][6][3]
    const T* pv;        // [KP_COUNT][n] or nullptr
    T* traj;            // snapshot s (global step (s+1)*stride) at traj[(s - snap_base)*n*NX ...] or nullptr
    T* mincos;          // [n] running min of |cos theta| (in/out) or nullptr
    T* gen_snap;        // generated inputs: AR(1) state before local step gen_snap_step is stored here ([n][NU]) or nullptr
    Health health;      // counters == nullptr: off
    long long snap_base;
    long long step0;    // global index of the first step of this launch
    int n, steps, stride;
    int u_vec, traj_vec;
    int lag_in_w;       // lag_in holds allocation-projected states [n][6][3]
    int mincos_init;    // 1: ignore the incoming mincos values (first chunk)
    int gen_snap_step;
    // Temporal tiling against wave quantisation (see rollout_kernel): the launch is cut into `quanta` time slices
    // per vehicle block; blocks take (slice, vehicle-block) work items from `ticket` in slice-major order and wait on
    // `progress[vehicle-block]` for their predecessor slice.  quanta <= 1: plain one-block-per-vehicle-block launch.
    int quanta;
    int nvblocks;       // vehicle blocks = ceil(n / BLOCK)
    int* ticket;        // [1], zero before the launch
    int* progress;      // [nvblocks], zero before the launch
};

template <typename T> struct RhsArgs {
    Consts<T> c;
    const T* x;
    const T* u;
    T* lag;    // in/out, nullptr = zero lag, not written
    const T* pv;
    T* xdot;
    int n;
};

template <typename T> struct SeArgs {
    Consts<T> c;
    const T* X;     // [rows][NX]
    const T* U;     // [rows][NU]
    const T* lag0;  // [nwin][NLAG] or nullptr
    double* partial;  // [gridDim.x][MAX_H]
    int rows, nwin, nH;
    int H[MAX_H];   // ascending
    // lag carry (thruster model, one horizon): window k starts from the lag state the reference's single model object
    // holds after windows 0..k-1 (SURVEY trap T3).  The lag is a stable linear filter, so only the last carry_steps
    // integrator steps of that history are distinguishable from zero in floating point; each thread replays them.
    int carry_steps;      // 0 = off
    // windows per thread.  Carried-lag mode: a thread that scores consecutive windows hands its lag from one to the
    // next for free (the end of window k IS the start of window k+1 for the shared model object) and pays the replay
    // once per wpt windows instead of once per window (49 replayed steps against H = 1 or 10 of its own).
    int wpt;
    long long win0;       // global index of local window 0
    long long row0;       // global index of local row 0 of X / U
    Health health;        // windows with a non-finite endpoint error / that came within eps of the singularity
    // Temporal tiling (reset mode, wpt = 1), as in rollout_kernel: the longest horizon is cut into `quanta` slices,
    // blocks take (slice, window-block) items from `ticket` in slice-major order and wait on `progress[window-block]`
    // for their predecessor; state, lag, min |cos theta| and the non-finite flag pass through the st_* scratch rows.
    // 125,000 windows per GPU (the 8-GPU shard of the 1M-window series) are 977 blocks on 296 slots: 4 rounds of 100
    // steps for 3.3 rounds of work; with 3 slices 10 rounds of 34.
    int quanta;           // <= 1: plain launch
    int nwblocks;         // window blocks (= gridDim.x / quanta)
    int* ticket;          // [1], zero before the launch
    int* progress;        // [nwblocks], zero before the launch
    T* st_x;              // [nwin][NX]
    T* st_lag;            // [nwin][18]
    float* st_mc;         // [nwin]
    int* st_bad;          // [nwin]
};

// ---------------------------------------------------------------------------------------------------------------
// vectorised, cache-hinted input loads
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int NU, bool STREAM>
__device__ __forceinline__ void load_u(const T* __restrict__ p, bool vec, T* __restrict__ u) {
    if (vec) {
        if constexpr (sizeof(T) == 4 && NU == 8) {
            const float4* q = reinterpret_cast<const float4*>(p);
            float4 a = STREAM ? __ldcs(q) : __ldg(q);
            float4 b = STREAM ? __ldcs(q + 1) : __ldg(q + 1);
            u[0] = a.x; u[1] = a.y; u[2] = a.z; u[3] = a.w; u[4] = b.x; u[5] = b.y; u[6] = b.z; u[7] = b.w;
        } else if constexpr (sizeof(T) == 4) {
            const float2* q = reinterpret_cast<const float2*>(p);
#pragma unroll
            for (int i = 0; i < NU / 2; ++i) {
                float2 a = STREAM ? __ldcs(q + i) : __ldg(q + i);
                u[2 * i] = a.x; u[2 * i + 1] = a.y;
            }
        } else {
            const double2* q = reinterpret_cast<const double2*>(p);
#pragma unroll
            for (int i = 0; i < NU / 2; ++i) {
                double2 a = STREAM ? __ldcs(q + i) : __ldg(q + i);
                u[2 * i] = a.x; u[2 * i + 1] = a.y;
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < NU; ++i) u[i] = STREAM ? __ldcs(p + i) : __ldg(p + i);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// trajectory snapshot: registers -> per-warp shared-memory tile [32][NX] -> 128-bit coalesced streaming stores
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int NX>
__device__ __forceinline__ void snapshot_warp(T* __restrict__ tile, const T* __restrict__ x, T* __restrict__ dst,
                                              int n_valid, bool vec, int lane) {
#pragma unroll
    for (int j = 0; j < NX; ++j) tile[lane * NX + j] = x[j];
    __syncwarp();
    constexpr int VEC = 16 / sizeof(T);
    if (vec) {
        using V = typename std::conditional<sizeof(T) == 4, float4, double2>::type;
#pragma unroll
        for (int e = 0; e < 32 * NX; e += 32 * VEC) {
            int idx = e + lane * VEC;
            if (idx + VEC <= n_valid) {
                __stcs(reinterpret_cast<V*>(dst + idx), *reinterpret_cast<const V*>(tile + idx));
            } else {
#pragma unroll
                for (int t = 0; t < VEC; ++t)
                    if (idx + t < n_valid) __stcs(dst + idx + t, tile[idx + t]);
            }
        }
    } else {
        for (int idx = lane; idx < n_valid; idx += 32) __stcs(dst + idx, tile[idx]);
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// rollout
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int MODEL, bool LAG1> struct LagRegs {
    static constexpr int N = (MODEL == MODEL_THRUSTER8) ? 18 : (LAG1 ? 6 : 1);
    static constexpr bool HAS = (MODEL == MODEL_THRUSTER8) || LAG1;
};

// Loads the lag state of vehicle i into registers; a per-thruster state [8][3] is projected on the way in.
template <typename T, int MODEL, bool LAG1>
__device__ __forceinline__ void load_lag(const Consts<T>& c, const T* __restrict__ src, bool src_is_w, long long i,
                                         T* __restrict__ lag) {
    constexpr int NL = LagRegs<T, MODEL, LAG1>::N;
    if (!LagRegs<T, MODEL, LAG1>::HAS || src == nullptr) {
#pragma unroll
        for (int j = 0; j < NL; ++j) lag[j] = T(0);
        return;
    }
    if constexpr (MODEL == MODEL_THRUSTER8) {
        if (src_is_w) {
#pragma unroll
            for (int j = 0; j < 18; ++j) lag[j] = __ldcg(src + i * 18 + j);
        } else {
            T t[24];
#pragma unroll
            for (int j = 0; j < 24; ++j) t[j] = __ldcg(src + i * 24 + j);
            project_lag<T>(c, t, lag);
        }
    } else {
#pragma unroll
        for (int j = 0; j < NL; ++j) lag[j] = __ldcg(src + i * NL + j);
    }
}

template <typename T> __device__ __forceinline__ bool finite_(T v) { return abs_(v) <= (sizeof(T) == 8 ? T(1.7976931348623157e308) : T(3.4028234663852886e38)); }

// warp-aggregated health counters: one atomic per warp and counter
__device__ __forceinline__ void count_health(const Health& h, bool bad, bool near_singular, int lane) {
    const unsigned bm = __ballot_sync(0xffffffffu, bad), sm = __ballot_sync(0xffffffffu, near_singular);
    if (lane == 0) {
        if (bm) atomicAdd(h.counters + 0, (unsigned long long)__popc(bm));
        if (sm) atomicAdd(h.counters + 1, (unsigned long long)__popc(sm));
    }
}

// GEN: the inputs are generated in the kernel (gen_advance) instead of being read from a.U
template <typename T, int MODEL, int INTEG, bool LAG1, bool PV, bool GEN, bool CU>
__global__ void __launch_bounds__(ROLLOUT_BLOCK) __maxnreg__(MaxReg<T>::N)
rollout_kernel(const __grid_constant__ RolloutArgs<T> a) {
    constexpr int BLOCK = ROLLOUT_BLOCK;
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    using LR = LagRegs<T, MODEL, LAG1>;
    constexpr int NL = LR::N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* smem = reinterpret_cast<T*>(smem_raw);

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;

    // Work item of this block.  Plain launch: vehicle block = blockIdx.x, all steps.  Temporal tiling: vehicles are
    // independent but a launch of B vehicle blocks on S resident slots costs ceil(B/S) rounds of the FULL step
    // count (65,536 fp64 vehicles: 512 blocks on 296 slots = 2 rounds for 1.73 rounds of work).  Cutting the steps
    // into Q slices turns that into ceil(B*Q/S) rounds of steps/Q (Q = 4: 7 rounds of 25 instead of 2 of 100).
    // Items are handed out by an atomic ticket in slice-major order, so the predecessor slice of a vehicle block
    // was always claimed earlier by a block that is resident and will finish: the wait below cannot deadlock.
    int vb = blockIdx.x, slice = 0;
    int k_begin = 0, k_end = a.steps;
    if (a.quanta > 1) {
        __shared__ int s_item;
        if (tid == 0) s_item = atomicAdd(a.ticket, 1);
        __syncthreads();
        // the ticket is the same for every thread of the block; passing it through a warp reduction lets the compiler
        // see that (REDUX writes a uniform register), so slice bounds and the step loop run on the uniform datapath
        const int item = __reduce_max_sync(0xffffffffu, s_item);
        slice = item / a.nvblocks;
        vb = item - slice * a.nvblocks;
        const int per = (a.steps + a.quanta - 1) / a.quanta;
        k_begin = slice * per;
        k_end = k_begin + per < a.steps ? k_begin + per : a.steps;
        if (slice > 0) {
            if (tid == 0) {
                const volatile int* flag = a.progress + vb;
                while (*flag < slice) __nanosleep(200);
                __threadfence();
            }
            __syncthreads();
        }
    }
    const long long gi = (long long)vb * BLOCK + tid;
    const bool live = gi < a.n;
    const long long i = live ? gi : (long long)a.n - 1;  // dead lanes shadow the last vehicle, never store

    // fp64: the constant block is staged into shared memory and read from there: sm_100 feeds FP instructions from
    // uniform registers, and the ~130 64-bit constants of a step do not fit them (kernel-argument operands end up
    // hoisted into regular registers and shuffled back through R2UR / UMOV: 0.491 against 0.481 ms, r01e)
    constexpr bool CSM = sizeof(T) == 8;
    __shared__ __align__(16) unsigned char cs_raw[CSM ? sizeof(Consts<T>) : 16];
    if constexpr (CSM) {
        const T* src = reinterpret_cast<const T*>(&a.c);
        T* dst = reinterpret_cast<T*>(cs_raw);
        for (int j = tid; j < (int)(sizeof(Consts<T>) / sizeof(T)); j += BLOCK) dst[j] = src[j];
        __syncthreads();
    }
    const Consts<T>& cc = CSM ? *reinterpret_cast<const Consts<T>*>(cs_raw) : a.c;

    // per-vehicle (Monte-Carlo) coefficients: registers (fp32) or a shared-memory table [36][BLOCK] (fp64)
    constexpr bool PVR = PvInRegs<T, PV>::V;
    typename std::conditional<PVR, ParamsRegs<T>,
                              typename std::conditional<PV, ParamsShared<T>, ParamsConst<T>>::type>::type p;
    if constexpr (PVR) {
#pragma unroll
        for (int j = 0; j < KP_COUNT; ++j) p.v[j] = __ldg(a.pv + (long long)j * a.n + i);
    } else if constexpr (PV) {
#pragma unroll 4
        for (int j = 0; j < KP_COUNT; ++j) smem[j * BLOCK + tid] = __ldg(a.pv + (long long)j * a.n + i);
        p.base = smem + tid;
        p.pitch = BLOCK;
        smem += KP_COUNT * BLOCK;
        __syncthreads();
    } else {
        p.kp = cc.kp;
    }
    T* tiles = smem;

    // slice 0 starts from (x0, lag_in); later slices continue from what the predecessor left in (xT, lag_out).
    // L2-only loads: another SM may have written these lines during this launch.
    const T* xsrc = slice > 0 ? a.xT : a.x0;
    T x[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) x[j] = __ldcg(xsrc + i * NX + j);
    T lag[NL];
    if (slice > 0) load_lag<T, MODEL, LAG1>(a.c, a.lag_out, true, i, lag);
    else load_lag<T, MODEL, LAG1>(a.c, a.lag_in, a.lag_in_w != 0, i, lag);
    float mc = 1.0f;   // running min of |cos theta| (float: a health metric, and one register in the fp64 kernels)
    if (a.mincos && (slice > 0 || !a.mincos_init)) mc = (float)__ldcg(a.mincos + i);

    const int nsteps = k_end - k_begin;
    const long long warp_v0 = (long long)vb * BLOCK + warp * 32;
    const long long rem = (long long)a.n - warp_v0;
    const int warp_n = (int)(rem < 0 ? 0 : (rem > 32 ? 32 : rem));   // live vehicles of this warp
    const int n_valid = warp_n * NX;

    // Inputs of the step, one of two sources:
    //  GEN       generated in the kernel: gs is the AR(1) state of the command signal, the deviates of the next step
    //            are drawn between the stages of the current one (GenSide);
    //  prefetch  any layout: the next step's row is requested into registers between stages 2 and 3 of the current
    //            step (LateSide).
    T u[NU];
    constexpr bool PREFETCH = !GEN;
    const T* up = a.U + i * a.u_stride_n + (long long)k_begin * a.u_stride_t;
    const bool uvec = a.u_vec != 0;
    const bool stream = a.u_stride_n != 0;  // per-vehicle inputs are read exactly once: evict-first
    float gs[GEN ? NU : 1];
    if constexpr (GEN) {
        const T* ssrc = slice > 0 ? a.gen.state_out : a.gen.state_in;
#pragma unroll
        for (int j = 0; j < NU; ++j) gs[j] = ssrc ? (float)__ldcg(ssrc + i * NU + j) : 0.0f;
    } else if (nsteps > 0) {
        if (stream) load_u<T, NU, true>(up, uvec, u); else load_u<T, NU, false>(up, uvec, u);
    }

    const long long gstep0 = a.step0 + k_begin;
    const unsigned long long veh = a.gen.vehicle0 + (unsigned long long)i;
    int countdown = a.traj ? (int)(a.stride - (gstep0 % a.stride)) : 0x7fffffff;
    long long snap = a.traj ? (gstep0 / a.stride - a.snap_base) : 0;
    // generated inputs: gs enters every step as the state that step uses; the prologue advances the state handed in
    // (the one before the first step) once, the steps advance it for their successors (GenSide)
    float gs_dummy[1];
    typename std::conditional<GEN, GenSide<T, NU>, NoSide>::type side{a.gen, GEN ? gs : gs_dummy};
    if constexpr (GEN) {
        if (nsteps > 0) { side.start(veh, gstep0, true); side.all(); }
    }

    for (int k = 0; k < nsteps; ++k) {
        T un[PREFETCH ? NU : 1];
        if constexpr (GEN) {
            // the state BEFORE step gen_snap_step is the one this step uses when it is that step's predecessor
            if (a.gen_snap && k_begin + k + 1 == a.gen_snap_step && live) {
#pragma unroll
                for (int j = 0; j < NU; ++j) a.gen_snap[i * NU + j] = T(gs[j]);
            }
#pragma unroll
            for (int j = 0; j < NU; ++j) u[j] = T(gs[j]);
            side.start(veh, gstep0 + k + 1, k + 1 < nsteps);
        }

        T acth;
        if constexpr (PREFETCH) {   // the next step's row is requested between stages 2 and 3 (LateSide)
            const T* nxt = up + (long long)((k + 1 < nsteps) ? (k + 1) : k) * a.u_stride_t;
            // CU = false is the build for the common case — no ocean current AND aligned per-vehicle input rows — with
            // the layout decided at compile time as well: no branch at the prefetch point in the middle of the step
            // (+1 %, r02t batch 7; not for the fp64 Monte-Carlo kernels, which lose 4 % with it)
            constexpr bool FASTU = !CU && !(PV && sizeof(T) == 8);
            auto pf = [&]() {
                if constexpr (FASTU) load_u<T, NU, true>(nxt, true, un);
                else if (stream) load_u<T, NU, true>(nxt, uvec, un);
                else load_u<T, NU, false>(nxt, uvec, un);
            };
            LateSide<decltype(pf)> late{pf, 1};
            integrate_step<T, MODEL, INTEG, LAG1, decltype(p), decltype(late), CU>(cc, p, x, lag, u, acth, late);
        } else {
            integrate_step<T, MODEL, INTEG, LAG1, decltype(p), decltype(side), CU>(cc, p, x, lag, u, acth, side);
        }
        mc = fminf(mc, (float)acth);

        if (--countdown == 0) {
            countdown = a.stride;
            T* dst = a.traj + (snap * a.n + warp_v0) * NX;
            snapshot_warp<T, NX>(tiles + warp * 32 * NX, x, dst, n_valid, a.traj_vec != 0, lane);
            ++snap;
        }
        if constexpr (PREFETCH) {
#pragma unroll
            for (int j = 0; j < NU; ++j) u[j] = un[j];
        }
    }

    if (live) {
#pragma unroll
        for (int j = 0; j < NX; ++j) a.xT[i * NX + j] = x[j];
        if (LR::HAS && a.lag_out) {
#pragma unroll
            for (int j = 0; j < NL; ++j) a.lag_out[i * NL + j] = lag[j];
        }
        if (a.mincos) a.mincos[i] = T(mc);
        if constexpr (GEN) {
            if (a.gen.state_out) {
#pragma unroll
                for (int j = 0; j < NU; ++j) a.gen.state_out[i * NU + j] = T(gs[j]);
            }
        }
    }
    if (a.health.counters && (a.quanta <= 1 || slice == a.quanta - 1)) {
        bool bad = false;
#pragma unroll
        for (int j = 0; j < NX; ++j) bad |= !finite_(x[j]);
        count_health(a.health, live && bad, live && ((double)mc < a.health.eps), lane);
    }
    if (a.quanta > 1) {  // publish this slice: state stores first, then the flag
        __threadfence();
        __syncthreads();
        if (tid == 0) atomicExch(a.progress + vb, slice + 1);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// per-thruster lag states after a rollout (thruster model): ThrusterLag._x of each thruster, [n][8][3]
// (fossen/BlueROV2.py:503-510).  The rollout kernel integrates the six allocation-projected filters; the per-thruster
// states are not recoverable from those, but each is a STABLE linear filter of its own thruster's input alone, so its
// state after the call is determined — to below one ulp — by the last `depth` inputs (brov_se_carry_steps: ||A^depth||
// < 1e-22) or, for a shorter call, by lag_in and all of them.  One thread per (vehicle, thruster) replays steps
// [first, steps): consecutive threads read consecutive scalars of the input rows and write consecutive triples.
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct LagTailArgs {
    Consts<T> c;
    InputGen<T> gen;        // gen.on: regenerate the inputs from gen_state (one thread per vehicle)
    const T* U;
    long long u_stride_t, u_stride_n;
    const T* lag_in;        // [n][8][3] state before step `first`, or nullptr = zeros
    T* lag_out;             // [n][8][3] (may alias lag_in)
    const T* gen_state;     // generated inputs: AR(1) state before step `first`, [n][8], or nullptr = zeros
    long long step0;
    int n, first, steps;
};

template <typename T>
__global__ void __launch_bounds__(TAIL_BLOCK) lag_tail_kernel(const __grid_constant__ LagTailArgs<T> a) {
    const long long g = (long long)blockIdx.x * TAIL_BLOCK + threadIdx.x;
    if (g >= (long long)a.n * 8) return;
    const long long i = g >> 3;
    const int t = (int)(g & 7);
    T x[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) x[j] = a.lag_in ? a.lag_in[g * 3 + j] : T(0);
    const T* up = a.U + i * a.u_stride_n + t;
    for (int k = a.first; k < a.steps; ++k) {
        const T F = thrust_poly<T>(__ldg(up + (long long)k * a.u_stride_t));
        lag_advance1<T>(a.c, x, F);
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) a.lag_out[g * 3 + j] = x[j];
}

template <typename T>
__global__ void __launch_bounds__(RHS_BLOCK) lag_tail_gen_kernel(const __grid_constant__ LagTailArgs<T> a) {
    const long long i = (long long)blockIdx.x * RHS_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    T lag[24];
    float s[8];
#pragma unroll
    for (int j = 0; j < 24; ++j) lag[j] = a.lag_in ? a.lag_in[i * 24 + j] : T(0);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = a.gen_state ? (float)a.gen_state[i * 8 + j] : 0.0f;
    const unsigned long long veh = a.gen.vehicle0 + (unsigned long long)i;
    for (int k = a.first; k < a.steps; ++k) {
        gen_advance<T, 8>(a.gen, veh, a.step0 + k, s);
        T F[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) F[j] = thrust_poly<T>(T(s[j]));
        lag_advance<T, false>(a.c, lag, F);
    }
#pragma unroll
    for (int j = 0; j < 24; ++j) a.lag_out[i * 24 + j] = lag[j];
}

// ---------------------------------------------------------------------------------------------------------------
// the generated command signal, materialised: U[k][j][:] for steps step0 .. step0+steps-1 and the selected vehicles
// first, first + vstride, ... (n_sel of them).  Same device function as the rollout kernels (gen_advance): a rollout
// fed with this array reproduces the generated-input rollout bit for bit, and the CPU oracle consumes the same values.
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct GenInputsArgs {
    InputGen<T> gen;        // state_in / state_out are indexed by SELECTED vehicle j: [n_sel][NU]
    T* out;                 // [steps][n_sel][NU]
    long long first, vstride, n_sel;
    long long step0;
    int steps;
};

template <typename T, int NU>
__global__ void __launch_bounds__(RHS_BLOCK) gen_inputs_kernel(const __grid_constant__ GenInputsArgs<T> a) {
    const long long j = (long long)blockIdx.x * RHS_BLOCK + threadIdx.x;
    if (j >= a.n_sel) return;
    const unsigned long long veh = a.gen.vehicle0 + (unsigned long long)(a.first + j * a.vstride);
    float s[NU];
#pragma unroll
    for (int q = 0; q < NU; ++q) s[q] = a.gen.state_in ? (float)a.gen.state_in[j * NU + q] : 0.0f;
    for (int k = 0; k < a.steps; ++k) {
        gen_advance<T, NU>(a.gen, veh, a.step0 + k, s);
#pragma unroll
        for (int q = 0; q < NU; ++q) a.out[((long long)k * a.n_sel + j) * NU + q] = T(s[q]);
    }
    if (a.gen.state_out) {
#pragma unroll
        for (int q = 0; q < NU; ++q) a.gen.state_out[j * NU + q] = T(s[q]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// single state-derivative evaluation (the reference's dynamics(): the 3rd-order lag advances by ONE sub-step)
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int MODEL, bool LAG1, bool PV>
__global__ void __launch_bounds__(RHS_BLOCK) rhs_kernel(const __grid_constant__ RhsArgs<T> a) {
    constexpr int BLOCK = RHS_BLOCK;
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    constexpr int NL = (MODEL == MODEL_THRUSTER8) ? 24 : (LAG1 ? 6 : 1);   // per-thruster lag states here
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* smem = reinterpret_cast<T*>(smem_raw);
    const int tid = threadIdx.x;
    const long long gi = (long long)blockIdx.x * BLOCK + tid;
    const bool live = gi < a.n;
    const long long i = live ? gi : (long long)a.n - 1;
    typename std::conditional<PV, ParamsShared<T>, ParamsConst<T>>::type p;
    if constexpr (PV) {
        for (int j = 0; j < KP_COUNT; ++j) smem[j * BLOCK + tid] = __ldg(a.pv + (long long)j * a.n + i);
        __syncthreads();
        p.base = smem + tid;
        p.pitch = BLOCK;
    } else {
        p.kp = a.c.kp;
    }
    T x[NX], u[NU], lag[NL], Fu[NU], xd[NX], lagd[6];
#pragma unroll
    for (int j = 0; j < NX; ++j) x[j] = __ldg(a.x + i * NX + j);
#pragma unroll
    for (int j = 0; j < NU; ++j) u[j] = __ldg(a.u + i * NU + j);
#pragma unroll
    for (int j = 0; j < NL; ++j) lag[j] = (LagRegs<T, MODEL, LAG1>::HAS && a.lag) ? a.lag[i * NL + j] : T(0);
#pragma unroll
    for (int j = 0; j < NU; ++j) Fu[j] = (MODEL == MODEL_THRUSTER8) ? thrust_poly<T>(u[j]) : u[j];
    if constexpr (ModelDim<MODEL>::DI) di_accel<T, NU>(a.c, u, Fu);
    Trig<T> tr;
    if constexpr (!ModelDim<MODEL>::QUAT) trig_full<T>(x + 3, tr);
    model_rhs<T, MODEL, LAG1, false, decltype(p)>(a.c, p, 0, x, tr, lag, Fu, xd, lagd);
    if (!live) return;
#pragma unroll
    for (int j = 0; j < NX; ++j) a.xdot[i * (NX + (LAG1 ? 6 : 0)) + j] = xd[j];
    if constexpr (LAG1) {
#pragma unroll
        for (int j = 0; j < 6; ++j) a.xdot[i * (NX + 6) + NX + j] = lagd[j];
    }
    if constexpr (MODEL == MODEL_THRUSTER8) {
        if (a.lag) {
            lag_advance<T, false>(a.c, lag, Fu);
#pragma unroll
            for (int j = 0; j < NL; ++j) a.lag[i * NL + j] = lag[j];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// thruster map alone: voltages -> polynomial -> one lag step -> body wrench   (compute_thruster_forces,
// fossen/BlueROV2.py:265-278; stateful like the reference)
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct ThrusterArgs {
    Consts<T> c;
    const T* u;   // [n][8]
    T* lag;       // [n][24] in/out or nullptr
    T* tau;       // [n][6]
    int n;
};

template <typename T>
__global__ void __launch_bounds__(RHS_BLOCK) thruster_wrench_kernel(const __grid_constant__ ThrusterArgs<T> a) {
    const long long i = (long long)blockIdx.x * RHS_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    T u[8], F[8], lag[24], tau[6];
    load_u<T, 8, false>(a.u + i * 8, (reinterpret_cast<uintptr_t>(a.u) & 15) == 0, u);
#pragma unroll
    for (int j = 0; j < 8; ++j) F[j] = thrust_poly<T>(u[j]);
#pragma unroll
    for (int j = 0; j < 24; ++j) lag[j] = a.lag ? a.lag[i * 24 + j] : T(0);
    thruster_tau<T, false>(a.c, 0, lag, F, tau);
#pragma unroll
    for (int j = 0; j < 6; ++j) a.tau[i * 6 + j] = tau[j];
    if (a.lag) {
        lag_advance<T, false>(a.c, lag, F);
#pragma unroll
        for (int j = 0; j < 24; ++j) a.lag[i * 24 + j] = lag[j];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// thruster map along a recorded input series with ONE carried lag state — what a loop over
// rov.compute_thruster_forces(U[k], dt) produces (make_pinc_dataset, training/train_tank_brov2_rk4.py:676-696).  The lag
// is a stable linear filter of the inputs only, so row k depends on the last `depth` rows to below one ulp: one thread
// per row replays them (rows are independent, the series is scored in parallel).
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct ThrusterSeriesArgs {
    Consts<T> c;
    const T* U;        // [rows][8]
    const T* lag0;     // [8][3] state before row 0, or nullptr (zeros)
    T* tau;            // [rows][6]
    T* lag_end;        // [8][3] state after the last row, or nullptr
    long long rows;
    int depth;
};

template <typename T>
__global__ void __launch_bounds__(RHS_BLOCK) thruster_series_kernel(const __grid_constant__ ThrusterSeriesArgs<T> a) {
    const long long k = (long long)blockIdx.x * RHS_BLOCK + threadIdx.x;
    if (k >= a.rows) return;
    T lag[24];
    const long long first = (k >= a.depth) ? k - a.depth : 0;
#pragma unroll
    for (int j = 0; j < 24; ++j) lag[j] = (first == 0 && a.lag0) ? a.lag0[j] : T(0);
    const bool vec = (reinterpret_cast<uintptr_t>(a.U) & 15) == 0;
    T u[8], F[8];
    for (long long r = first; r < k; ++r) {
        load_u<T, 8, false>(a.U + r * 8, vec, u);
#pragma unroll
        for (int j = 0; j < 8; ++j) F[j] = thrust_poly<T>(u[j]);
        lag_advance<T, false>(a.c, lag, F);
    }
    load_u<T, 8, false>(a.U + k * 8, vec, u);
#pragma unroll
    for (int j = 0; j < 8; ++j) F[j] = thrust_poly<T>(u[j]);
    T tau[6];
    thruster_tau<T, false>(a.c, 0, lag, F, tau);
#pragma unroll
    for (int j = 0; j < 6; ++j) a.tau[k * 6 + j] = tau[j];
    if (a.lag_end && k == a.rows - 1) {
        lag_advance<T, false>(a.c, lag, F);
#pragma unroll
        for (int j = 0; j < 24; ++j) a.lag_end[j] = lag[j];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// multi-horizon endpoint squared error over sliding windows
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int MODEL, int INTEG>
__global__ void __launch_bounds__(ROLLOUT_BLOCK) __maxnreg__(MaxReg<T>::N)
se_kernel(const __grid_constant__ SeArgs<T> a) {
    constexpr int BLOCK = ROLLOUT_BLOCK;
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    // the evaluator never returns lag states: the thruster model runs on the allocation-projected lag
    using LR = LagRegs<T, MODEL, false>;
    constexpr int NL = LR::N;
    __shared__ double red[BLOCK / 32][MAX_H];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int hmax = a.H[a.nH - 1];
    // work item: window block wb, steps [j_begin, j_end) of its windows (temporal tiling, see SeArgs::quanta)
    int wb = blockIdx.x, slice = 0, j_begin = 0, j_end = hmax;
    if (a.quanta > 1) {
        __shared__ int s_item;
        if (tid == 0) s_item = atomicAdd(a.ticket, 1);
        __syncthreads();
        const int item = __reduce_max_sync(0xffffffffu, s_item);
        slice = item / a.nwblocks;
        wb = item - slice * a.nwblocks;
        const int per = (hmax + a.quanta - 1) / a.quanta;
        j_begin = slice * per;
        j_end = j_begin + per < hmax ? j_begin + per : hmax;
        if (slice > 0) {
            if (tid == 0) {
                const volatile int* flag = a.progress + wb;
                while (*flag < slice) __nanosleep(200);
                __threadfence();
            }
            __syncthreads();
        }
    }
    const bool last_slice = slice >= a.quanta - 1;
    // a thread scores a.wpt consecutive windows (1 except in carried-lag mode, see SeArgs::wpt)
    const long long gk = ((long long)wb * BLOCK + tid) * a.wpt;
    ParamsConst<T> p;
    p.kp = a.c.kp;
    const bool uvec = ((reinterpret_cast<uintptr_t>(a.U) & 15) == 0) && (sizeof(T) * NU % 16 == 0);
    double se[MAX_H];
#pragma unroll
    for (int h = 0; h < MAX_H; ++h) se[h] = 0.0;
    int n_bad = 0, n_sing = 0;
    T lag[NL];
    for (int c = 0; c < a.wpt; ++c) {
        const long long k = gk + c;
        if (k >= a.nwin) break;
        const long long kr = k + (a.win0 - a.row0);  // local row of the window's start (rows before it: carry history)
        T x[NX];
        if (slice > 0) {   // continue from what the predecessor slice left (L2-only loads: written during this launch)
#pragma unroll
            for (int j = 0; j < NX; ++j) x[j] = __ldcg(a.st_x + k * NX + j);
#pragma unroll
            for (int j = 0; j < NL; ++j) lag[j] = __ldcg(a.st_lag + k * 18 + j);
        } else {
#pragma unroll
            for (int j = 0; j < NX; ++j) x[j] = __ldg(a.X + kr * NX + j);
        }
        if (c == 0 && slice == 0) {
            load_lag<T, MODEL, false>(a.c, a.lag0, false, k, lag);
            if constexpr (MODEL == MODEL_THRUSTER8) {
                if (a.carry_steps > 0) {
                    // history of the shared model object: windows w = 0..kg-1, each feeding U[w..w+H-1]; replay its tail
                    const long long H0 = a.H[0];
                    const long long total = (a.win0 + k) * H0;
                    const long long m = total < a.carry_steps ? total : a.carry_steps;
                    for (long long s = total - m; s < total; ++s) {
                        const long long w = s / H0;
                        const long long row = w + (s - w * H0) - a.row0;
                        T u[NU], F[8], TF[6];
                        load_u<T, NU, false>(a.U + row * NU, uvec, u);
#pragma unroll
                        for (int i = 0; i < 8; ++i) F[i] = thrust_poly<T>(u[i]);
                        allocate_wrench<T>(a.c, F, TF);
                        lag_advance<T, true>(a.c, lag, TF);
                    }
                }
            }
        }   // c > 0: the lag this thread's previous window ended with IS the state the shared object hands to this one

        // window k may run j steps while row k + j exists
        long long room = (long long)a.rows - 1 - kr;
        const int nsteps = (int)(room < hmax ? (room < 0 ? 0 : room) : hmax);
        float mc = 1.0f;
        bool bad = false;
        if (slice > 0) {
            mc = __ldcg(a.st_mc + k);
            bad = __ldcg(a.st_bad + k) != 0;
        }
        const int j_stop = nsteps < j_end ? nsteps : j_end;
        T u[NU], un[NU];
        if (j_begin < j_stop) load_u<T, NU, false>(a.U + (kr + j_begin) * NU, uvec, u);
        for (int j = j_begin; j < j_stop; ++j) {
            // the next step's input row is requested between stages 2 and 3 of this one (LateSide, as in the rollout)
            const T* nxt = a.U + (kr + (j + 1 < j_stop ? j + 1 : j)) * NU;
            auto pf = [&]() { load_u<T, NU, false>(nxt, uvec, un); };
            LateSide<decltype(pf)> late{pf, 1};
            T acth;
            integrate_step<T, MODEL, INTEG, false, decltype(p)>(a.c, p, x, lag, u, acth, late);
#pragma unroll
            for (int q = 0; q < NU; ++q) u[q] = un[q];
            mc = fminf(mc, (float)acth);
#pragma unroll
            for (int h = 0; h < MAX_H; ++h) {
                if (h < a.nH && j + 1 == a.H[h]) {
                    const T* tgt = a.X + (kr + j + 1) * NX;
                    double s = 0.0;
#pragma unroll
                    for (int q = 0; q < NX; ++q) {
                        double e = (double)x[q] - (double)__ldg(tgt + q);
                        s += e * e;
                    }
                    se[h] += s;
                    bad |= !(s <= 1.7976931348623157e308);
                }
            }
        }
        if (last_slice) {
            n_bad += bad ? 1 : 0;
            n_sing += ((double)mc < a.health.eps) ? 1 : 0;
        } else {
#pragma unroll
            for (int j = 0; j < NX; ++j) a.st_x[k * NX + j] = x[j];
#pragma unroll
            for (int j = 0; j < NL; ++j) a.st_lag[k * 18 + j] = lag[j];
            a.st_mc[k] = mc;
            a.st_bad[k] = bad ? 1 : 0;
        }
    }
    if (!last_slice) {   // hand the window block to its next slice
        __threadfence();
        __syncthreads();
        if (tid == 0) atomicExch(a.progress + wb, slice + 1);
    }
    if (a.health.counters) {
        const int tb = __reduce_add_sync(0xffffffffu, n_bad), ts = __reduce_add_sync(0xffffffffu, n_sing);
        if (lane == 0) {
            if (tb) atomicAdd(a.health.counters + 0, (unsigned long long)tb);
            if (ts) atomicAdd(a.health.counters + 1, (unsigned long long)ts);
        }
    }
#pragma unroll
    for (int h = 0; h < MAX_H; ++h) {
        double v = se[h];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[warp][h] = v;
    }
    __syncthreads();
    if (tid < MAX_H) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < BLOCK / 32; ++w) v += red[w][tid];
        a.partial[((long long)slice * (a.quanta > 1 ? a.nwblocks : 0) + wb) * MAX_H + tid] = v;
    }
}

// one block; thread t sums partials t, t+256, ... in order, then a fixed tree: same bits every run
static __global__ void __launch_bounds__(256) se_finish_kernel(const double* __restrict__ partial, int nblocks,
                                                        double* __restrict__ se_out) {
    __shared__ double sh[256];
    for (int h = 0; h < MAX_H; ++h) {
        double v = 0.0;
        for (int b = threadIdx.x; b < nblocks; b += 256) v += partial[(long long)b * MAX_H + h];
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
            __syncthreads();
        }
        if (threadIdx.x == 0) se_out[h] = sh[0];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// candidate sweep: the endpoint squared error of P coefficient sets against ONE recorded series in one launch
// (calibration, sensitivity studies, scoring a Monte-Carlo cloud of vehicles).  A block is one item (candidate c,
// window block wb of ROLLOUT_BLOCK consecutive windows); its body is se_kernel's reset mode with one window per
// thread, so a candidate's sums equal those of brov_multistep_se(time_slices = 1) with that candidate's coefficients.
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct SweepArgs {
    Consts<T> c;        // engine constants (allocation, lag discretisation, dt, has_current); c.kp is not read
    const T* X;         // [rows][NX]
    const T* U;         // [rows][NU]
    const T* kp;        // [KP_COUNT][P] candidate coefficient table
    const T* lag0;      // per-window initial lag or nullptr (zeros): [nwin][24] (projected on load) or [nwin][18]
    int lag0_w;         // lag0 holds allocation-projected states [nwin][18] (carry mode: se_carry_lag_kernel's output)
    double* partial;    // [P][nwb][MAX_H]
    unsigned long long* health;   // [P][2] (non-finite, near-singular windows) or nullptr; zeroed before the launch
    double eps;
    long long off;      // local row of window 0 (window0 - row0)
    int rows, nwin, nH;
    int H[MAX_H];       // ascending
    int P, nwb;         // candidates, window blocks
};

// Item order: window-block-major (item = wb * P + c): the blocks resident at one time read the same few X / U rows,
// which L2 serves to all candidates.  Candidate-major (item = c * nwb + wb, BROV_SWEEP_CAND_MAJOR=1) measured the same
// on B200 within run-to-run noise (profiles/sweep_timing*.json: the build timed second was 2 % faster on the 1M-row
// series whichever order it had).
#ifndef BROV_SWEEP_CAND_MAJOR
#define BROV_SWEEP_CAND_MAJOR 0
#endif
// Candidate coefficients: staged once per block into shared memory and read as broadcasts (ParamsShared, pitch 1), so
// the kernel holds no per-thread table.  fp32 copies in registers (ParamsRegs, as the fp32 Monte-Carlo rollout does;
// BROV_SWEEP_KP_REGS=1) measured the same within noise and take a larger stack frame (96 against 72 bytes).
#ifndef BROV_SWEEP_KP_REGS
#define BROV_SWEEP_KP_REGS 0
#endif

template <typename T, int MODEL, int INTEG>
__global__ void __launch_bounds__(ROLLOUT_BLOCK) __maxnreg__(MaxReg<T>::N)
se_sweep_kernel(const __grid_constant__ SweepArgs<T> a) {
    constexpr int BLOCK = ROLLOUT_BLOCK;
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NU = ModelDim<MODEL>::NU;
    using LR = LagRegs<T, MODEL, false>;
    constexpr int NL = LR::N;
    __shared__ double red[BLOCK / 32][MAX_H];
    __shared__ T kps[KP_COUNT];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int hmax = a.H[a.nH - 1];
    const int item = blockIdx.x;
    const int cand = BROV_SWEEP_CAND_MAJOR ? item / a.nwb : item % a.P;
    const int wb = BROV_SWEEP_CAND_MAJOR ? item - cand * a.nwb : item / a.P;
    if (tid < KP_COUNT) kps[tid] = __ldg(a.kp + (long long)tid * a.P + cand);
    __syncthreads();
    constexpr bool KPR = BROV_SWEEP_KP_REGS && sizeof(T) == 4;
    typename std::conditional<KPR, ParamsRegs<T>, ParamsShared<T>>::type p;
    if constexpr (KPR) {
#pragma unroll
        for (int j = 0; j < KP_COUNT; ++j) p.v[j] = kps[j];
    } else {
        p.base = kps;
        p.pitch = 1;
    }
    const long long k = (long long)wb * BLOCK + tid;
    const bool uvec = ((reinterpret_cast<uintptr_t>(a.U) & 15) == 0) && (sizeof(T) * NU % 16 == 0);
    double se[MAX_H];
#pragma unroll
    for (int h = 0; h < MAX_H; ++h) se[h] = 0.0;
    int n_bad = 0, n_sing = 0;
    if (k < a.nwin) {
        const long long kr = k + a.off;
        T x[NX], lag[NL];
#pragma unroll
        for (int j = 0; j < NX; ++j) x[j] = __ldg(a.X + kr * NX + j);
        load_lag<T, MODEL, false>(a.c, a.lag0, a.lag0_w != 0, k, lag);
        // window k may run j steps while row k + j exists
        const long long room = (long long)a.rows - 1 - kr;
        const int nsteps = (int)(room < hmax ? (room < 0 ? 0 : room) : hmax);
        float mc = 1.0f;
        bool bad = false;
        T u[NU], un[NU];
        if (nsteps > 0) load_u<T, NU, false>(a.U + kr * NU, uvec, u);
        for (int j = 0; j < nsteps; ++j) {
            const T* nxt = a.U + (kr + (j + 1 < nsteps ? j + 1 : j)) * NU;
            auto pf = [&]() { load_u<T, NU, false>(nxt, uvec, un); };
            LateSide<decltype(pf)> late{pf, 1};
            T acth;
            integrate_step<T, MODEL, INTEG, false, decltype(p)>(a.c, p, x, lag, u, acth, late);
#pragma unroll
            for (int q = 0; q < NU; ++q) u[q] = un[q];
            mc = fminf(mc, (float)acth);
#pragma unroll
            for (int h = 0; h < MAX_H; ++h) {
                if (h < a.nH && j + 1 == a.H[h]) {
                    const T* tgt = a.X + (kr + j + 1) * NX;
                    double s = 0.0;
#pragma unroll
                    for (int q = 0; q < NX; ++q) {
                        double e = (double)x[q] - (double)__ldg(tgt + q);
                        s += e * e;
                    }
                    se[h] += s;
                    bad |= !(s <= 1.7976931348623157e308);
                }
            }
        }
        n_bad = bad ? 1 : 0;
        n_sing = ((double)mc < a.eps) ? 1 : 0;
    }
    if (a.health) {
        const int tb = __reduce_add_sync(0xffffffffu, n_bad), ts = __reduce_add_sync(0xffffffffu, n_sing);
        if (lane == 0) {
            if (tb) atomicAdd(a.health + 2 * cand + 0, (unsigned long long)tb);
            if (ts) atomicAdd(a.health + 2 * cand + 1, (unsigned long long)ts);
        }
    }
#pragma unroll
    for (int h = 0; h < MAX_H; ++h) {
        double v = se[h];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[warp][h] = v;
    }
    __syncthreads();
    if (tid < MAX_H) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < BLOCK / 32; ++w) v += red[w][tid];
        a.partial[((long long)cand * a.nwb + wb) * MAX_H + tid] = v;
    }
}

// one block per candidate, each the fixed-order sum of se_finish_kernel over that candidate's nwb partials
static __global__ void __launch_bounds__(256) se_sweep_finish_kernel(const double* __restrict__ partial, int nwb,
                                                                     double* __restrict__ se_out) {
    __shared__ double sh[256];
    partial += (long long)blockIdx.x * nwb * MAX_H;
    se_out += (long long)blockIdx.x * MAX_H;
    for (int h = 0; h < MAX_H; ++h) {
        double v = 0.0;
        for (int b = threadIdx.x; b < nwb; b += 256) v += partial[(long long)b * MAX_H + h];
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
            __syncthreads();
        }
        if (threadIdx.x == 0) se_out[h] = sh[0];
        __syncthreads();
    }
}

// Carried lag of the sweep (thruster model, one horizon H): the allocation-projected lag state [nwin][18] that window k
// inherits from windows 0..k-1 of the reference's single model object.  It depends on the inputs, dt, the integrator
// and the allocation only — never on the 36 coefficients — so one pass serves every candidate.  Same replay and
// window-to-window hand-over as se_kernel's carried-lag mode, with the dynamics left out: lag-only steps.
template <typename T> struct CarryLagArgs {
    Consts<T> c;
    const T* U;         // [rows][8]
    T* lag_out;         // [nwin][18]
    long long win0, row0;
    int rows, nwin, H, carry_steps, wpt;
};

template <typename T>
__global__ void __launch_bounds__(RHS_BLOCK) se_carry_lag_kernel(const __grid_constant__ CarryLagArgs<T> a) {
    const long long gk = ((long long)blockIdx.x * RHS_BLOCK + threadIdx.x) * a.wpt;
    const bool uvec = (reinterpret_cast<uintptr_t>(a.U) & 15) == 0;
    const long long H0 = a.H;
    T lag[18];
    for (int c = 0; c < a.wpt; ++c) {
        const long long k = gk + c;
        if (k >= a.nwin) break;
        const long long kr = k + (a.win0 - a.row0);
        T u[8], F[8], TF[6];
        if (c == 0) {
#pragma unroll
            for (int j = 0; j < 18; ++j) lag[j] = T(0);
            // history of the shared model object: windows w = 0..kg-1, each feeding U[w..w+H-1]; replay its tail
            const long long total = (a.win0 + k) * H0;
            const long long m = total < a.carry_steps ? total : a.carry_steps;
            for (long long s = total - m; s < total; ++s) {
                const long long w = s / H0;
                const long long row = w + (s - w * H0) - a.row0;
                load_u<T, 8, false>(a.U + row * 8, uvec, u);
#pragma unroll
                for (int i = 0; i < 8; ++i) F[i] = thrust_poly<T>(u[i]);
                allocate_wrench<T>(a.c, F, TF);
                lag_advance<T, true>(a.c, lag, TF);
            }
        }   // c > 0: the lag the previous window ended with IS the state the shared object hands to this one
#pragma unroll
        for (int j = 0; j < 18; ++j) a.lag_out[k * 18 + j] = lag[j];
        // window k: the lag advances once per step it runs (as in integrate_step)
        const long long room = (long long)a.rows - 1 - kr;
        const int nsteps = (int)(room < H0 ? (room < 0 ? 0 : room) : H0);
        for (int j = 0; j < nsteps; ++j) {
            load_u<T, 8, false>(a.U + (kr + j) * 8, uvec, u);
#pragma unroll
            for (int i = 0; i < 8; ++i) F[i] = thrust_poly<T>(a.c, u[i]);
            allocate_wrench<T>(a.c, F, TF);
            lag_advance<T, true>(a.c, lag, TF);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// reduced 9-state model RHS (bluerov_compute): 13 scalars in, 9 out per row; rows staged through shared memory so
// that every global access is a full-line coalesced (vector) transaction
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct Red9Consts {
    T im_u, im_v, im_w, im_r;   // 1/(m - X_ud), 1/(m - Y_vd), 1/(m - Z_wd), 1/(I_zz - N_rd)
    T mYv, mXu, dXY;            // m - Y_vd, m - X_ud, X_ud - Y_vd
    T Xu, Xuc, Yv, Yvc, Zw, Zwc, Nr, Nrc;
    T wnet;                     // m g - F_bouy
};

template <typename T>
__global__ void __launch_bounds__(RED9_BLOCK) reduced9_kernel(const __grid_constant__ Red9Consts<T> c,
                                                              const T* __restrict__ X, const T* __restrict__ U,
                                                              T* __restrict__ O, long long B, int vec) {
    __shared__ __align__(16) T tile[RED9_BLOCK * 9];
    constexpr int VEC = 16 / sizeof(T);
    using V = typename std::conditional<sizeof(T) == 4, float4, double2>::type;
    const int tid = threadIdx.x;
    const long long r0 = (long long)blockIdx.x * RED9_BLOCK;
    const long long rows = (B - r0 < RED9_BLOCK) ? (B - r0) : RED9_BLOCK;
    const int nel = (int)rows * 9;
    const T* src = X + r0 * 9;
    if (vec) {
        for (int e = tid * VEC; e < nel; e += RED9_BLOCK * VEC) {
            if (e + VEC <= nel) *reinterpret_cast<V*>(tile + e) = __ldcs(reinterpret_cast<const V*>(src + e));
            else for (int t = 0; e + t < nel; ++t) tile[e + t] = __ldcs(src + e + t);
        }
    } else {
        for (int e = tid; e < nel; e += RED9_BLOCK) tile[e] = __ldcs(src + e);
    }
    __syncthreads();
    T o[9];
    if (tid < rows) {
        const T* x = tile + tid * 9;  // stride 9 words: conflict-free
        T cps = x[3], sps = x[4], u = x[5], v = x[6], w = x[7], r = x[8];
        T in[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) in[j] = __ldcs(U + (r0 + tid) * 4 + j);
        o[0] = cps * u - sps * v;
        o[1] = sps * u + cps * v;
        o[2] = w;
        o[3] = -sps * r;
        o[4] = cps * r;
        o[5] = c.im_u * (in[0] + c.mYv * v * r + (c.Xu + c.Xuc * abs_(u)) * u);
        o[6] = c.im_v * (in[1] - c.mXu * u * r + (c.Yv + c.Yvc * abs_(v)) * v);
        o[7] = c.im_w * (in[2] + (c.Zw + c.Zwc * abs_(w)) * w + c.wnet);
        o[8] = c.im_r * (in[3] - c.dXY * u * v + (c.Nr + c.Nrc * abs_(r)) * r);
    }
    __syncthreads();
    if (tid < rows) {
#pragma unroll
        for (int j = 0; j < 9; ++j) tile[tid * 9 + j] = o[j];
    }
    __syncthreads();
    T* dst = O + r0 * 9;
    if (vec) {
        for (int e = tid * VEC; e < nel; e += RED9_BLOCK * VEC) {
            if (e + VEC <= nel) __stcs(reinterpret_cast<V*>(dst + e), *reinterpret_cast<const V*>(tile + e));
            else for (int t = 0; e + t < nel; ++t) __stcs(dst + e + t, tile[e + t]);
        }
    } else {
        for (int e = tid; e < nel; e += RED9_BLOCK) __stcs(dst + e, tile[e]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// FMA-chain microbenchmark: 8 independent chains per thread, 2 flops per FMA
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
    T v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = T(threadIdx.x + j) * T(1e-3);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = v[j] * a + b;
        }
    }
    T s = T(0);
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
    if (s == T(123456789)) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ---------------------------------------------------------------------------------------------------------------
// launchers (defined in brov_kernels_impl.cuh, instantiated per scalar type)
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
cudaError_t launch_rollout(int model, int integ, bool lag1, const RolloutArgs<T>& a, cudaStream_t st);
template <typename T> int rollout_blocks_per_sm(int model, int integ, bool lag1, bool pv, bool gen, bool traj, bool cur);
template <typename T> cudaError_t launch_lag_tail(const LagTailArgs<T>& a, cudaStream_t st);
template <typename T> cudaError_t launch_gen_inputs(int nu, const GenInputsArgs<T>& a, cudaStream_t st);
template <typename T>
cudaError_t launch_rhs(int model, bool lag1, const RhsArgs<T>& a, cudaStream_t st);
template <typename T>
cudaError_t launch_se(int model, int integ, const SeArgs<T>& a, double* se_out, cudaStream_t st);
template <typename T> int se_blocks(long long nwin);
template <typename T>
cudaError_t launch_se_sweep(int model, int integ, const SweepArgs<T>& a, double* se_out, cudaStream_t st);
template <typename T> cudaError_t launch_se_carry_lag(const CarryLagArgs<T>& a, cudaStream_t st);
template <typename T>
cudaError_t launch_reduced9(const Red9Consts<T>& c, const T* X, const T* U, T* O, long long B, cudaStream_t st);
template <typename T>
cudaError_t launch_fma_peak(int iters, int blocks, T* scratch, cudaStream_t st);
template <typename T>
cudaError_t launch_thruster_wrench(const ThrusterArgs<T>& a, cudaStream_t st);
template <typename T>
cudaError_t launch_thruster_series(const ThrusterSeriesArgs<T>& a, cudaStream_t st);

}  // namespace brov
