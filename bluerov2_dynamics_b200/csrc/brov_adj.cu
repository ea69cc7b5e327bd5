// brov_adj.cu — reverse-mode (adjoint) gradients of batched rollouts: for a loss L = sum_k <c_k, x_k> + <g_T, z_T> the
// kernels return dL/dz_0 and dL/du_k of every vehicle, with the step differentiated as brov_linearize differentiates
// it (full sines and cosines in every stage, branch taken, the quaternion renormalised after the step).
//
// One thread per vehicle, two loops in one launch.  The forward loop takes the primal steps from z_0 and stores every
// z_k in the workspace ([steps][NZ][n], coalesced).  The backward loop runs k = steps-1 .. 0: it reloads z_k, forms
// the step's input again, recomputes the stage states with the code the forward loop ran (so the map it
// differentiates is exactly the stored one), stages them in shared memory and sweeps the stages in reverse with the
// hand-written vector-Jacobian products of the right-hand sides (rhs_euler12_vjp / rhs_quat13_vjp, brov_device.cuh).
// The three kernels are built from the same pieces (adj_fwd_step, adj_step_vjp, adj_gu and the small I/O helpers):
//
//   adjoint_kernel              inputs U read from memory; stores dL/du_k.
//   adjoint_coef_kernel         adjoint_kernel's sweep, which also accumulates dL/dkp of the vehicle's coefficients.
//   closed_loop_adjoint_kernel  inputs from the in-kernel feedback law, reversed through the feedback after each step.
//
// Every sum has a fixed order, so the results are bit-reproducible and independent of the other vehicles.
#include "brov_adj.cuh"

#include <algorithm>
#include <type_traits>

namespace brov {

template <int MODEL> struct AdjDim {
    static constexpr int NX = LinDim<MODEL>::NX, NU = LinDim<MODEL>::NU, NZ = LinDim<MODEL>::NZ;
    static constexpr bool THR = MODEL == MODEL_THRUSTER8;
    static constexpr bool QUAT = ModelDim<MODEL>::QUAT;
    static constexpr int NL = THR ? 18 : 1;   // the thruster lag Z (one unused entry for the wrench models)
};

// Dynamic shared memory of the sweep kernels, in rows of ADJ_THREADS doubles (one column per thread, conflict-free):
// the RK4 stage buffer (3 NX rows) first, then `rows` more rows and `bytes` more bytes of the kernel's own
__host__ __device__ constexpr int adj_stage_rows(int model, int integ) {
    return integ == INTEG_RK4 ? 3 * (model == MODEL_QUAT13 ? 13 : 12) : 0;
}
constexpr size_t adj_smem_bytes(int model, int integ, int rows, size_t bytes) {
    return (size_t)(adj_stage_rows(model, integ) + rows) * ADJ_THREADS * sizeof(double) + bytes;
}

// right-hand side of sub-step s at the stage state xs, as linearize evaluates it (full sines and cosines)
template <int MODEL, class P>
__device__ __forceinline__ void adj_rhs(const Consts<double>& c, const P& p, int s, const double* __restrict__ xs,
                                        const double* __restrict__ Z, const double* __restrict__ Fw,
                                        double* __restrict__ out, double& abs_cth) {
    const bool cur = c.has_current != 0;
    double tau[6];
    if constexpr (MODEL == MODEL_THRUSTER8) {
        thruster_tau<double, true>(c, s, Z, Fw, tau);
    } else {
#pragma unroll
        for (int r = 0; r < 6; ++r) tau[r] = Fw[r];
    }
    if constexpr (!ModelDim<MODEL>::QUAT) {
        Trig<double> tr;
        trig_full<double>(c, xs + 3, tr);
        if (s == 0) abs_cth = fabs(tr.cth);
        rhs_euler12<double>(xs, tr, tau, p, cur, out);
    } else {
        rhs_quat13<double>(xs, tau, p, cur, out);
    }
}

// One primal step x <- Phi_x(x, Z, Fw); the lag is advanced by the caller.  STAGES (the backward loop's recompute): the
// RK4 stage states xs_1..xs_3 go to sx[((s-1)*NX + i) * ADJ_THREADS] and the quaternion before its renormalisation to
// qpre; the last stage's right-hand side is evaluated only when the renormalisation needs it.
template <int MODEL, int INTEG, bool STAGES, class P>
__device__ __forceinline__ void adj_step(const Consts<double>& c, const P& p, double* __restrict__ x, const double* __restrict__ Z,
                                         const double* __restrict__ Fw, double* __restrict__ sx,
                                         double* __restrict__ qpre, double& abs_cth) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr bool QUAT = ModelDim<MODEL>::QUAT;
    const double dt = c.dt;
    abs_cth = 1.0;
    double k[NX];
    if constexpr (INTEG == INTEG_EULER) {
        adj_rhs<MODEL>(c, p, 0, x, Z, Fw, k, abs_cth);
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt * k[i];
    } else {
        double acc[NX], xs[NX];
        const double hdt = 0.5 * dt;
        adj_rhs<MODEL>(c, p, 0, x, Z, Fw, k, abs_cth);
#pragma unroll
        for (int s = 1; s <= 3; ++s) {
            const double w = (s == 1) ? 1.0 : 2.0;
            const double h = (s == 3) ? dt : hdt;
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                if (s == 1) acc[i] = k[i]; else acc[i] += w * k[i];
                xs[i] = x[i] + h * k[i];
                if constexpr (STAGES) sx[((s - 1) * NX + i) * ADJ_THREADS] = xs[i];
            }
            if constexpr (STAGES && !QUAT) {
                if (s == 3) return;
            }
            adj_rhs<MODEL>(c, p, s, xs, Z, Fw, k, abs_cth);
        }
        const double dt6 = dt * (1.0 / 6.0);
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt6 * (acc[i] + k[i]);
    }
    if constexpr (QUAT) {
        if constexpr (STAGES) {
#pragma unroll
            for (int i = 0; i < 4; ++i) qpre[i] = x[3 + i];
        }
        quat_renorm<double>(x + 3);
    }
}

__device__ __forceinline__ bool adj_finite(double v) { return fabs(v) <= 1.7976931348623157e308; }

// ---- the pieces of the sweeps

// the wrench of the input row u: thruster8 through the thrust curve and the allocation, the wrench models u itself
template <int MODEL>
__device__ __forceinline__ void adj_wrench(const Consts<double>& c, const double* u, double* __restrict__ Fw) {
    if constexpr (MODEL == MODEL_THRUSTER8) {
        double F[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) F[i] = thrust_poly<double>(c, u[i]);
        allocate_wrench<double>(c, F, Fw);
    } else {
#pragma unroll
        for (int r = 0; r < 6; ++r) Fw[r] = u[r];
    }
}

// vehicle v's initial state from z0 [n][NZ]
template <int MODEL>
__device__ __forceinline__ void adj_load_z0(const double* z0, long long v, double* x, double* Z) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) x[q] = z0[v * D::NZ + q];
#pragma unroll
    for (int q = 0; q < D::NL; ++q) Z[q] = D::THR ? z0[v * D::NZ + D::NX + q] : 0.0;
}

// z_k to / from its slice wk of the workspace (vehicle index fastest)
template <int MODEL>
__device__ __forceinline__ void adj_store_z(double* wk, long long n, const double* x, const double* Z) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) wk[q * n] = x[q];
    if constexpr (D::THR) {
#pragma unroll
        for (int q = 0; q < D::NL; ++q) wk[(D::NX + q) * n] = Z[q];
    }
}
template <int MODEL>
__device__ __forceinline__ void adj_load_z(const double* wk, long long n, double* x, double* Z) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) x[q] = wk[q * n];
    if constexpr (D::THR) {
#pragma unroll
        for (int q = 0; q < D::NL; ++q) Z[q] = wk[(D::NX + q) * n];
    }
}

// forward step k from the input row u (z_k already stored): the wrench, the primal step, the singularity flag, the lag
template <int MODEL, int INTEG, class P>
__device__ __forceinline__ void adj_fwd_step(const Consts<double>& c, const P& p, double* x, double* Z, const double* u,
                                             double eps, bool& sing) {
    double Fw[6];
    adj_wrench<MODEL>(c, u, Fw);
    double acth;
    adj_step<MODEL, INTEG, false>(c, p, x, Z, Fw, nullptr, nullptr, acth);
    sing |= acth < eps;
    if constexpr (MODEL == MODEL_THRUSTER8) lag_advance<double, true>(c, Z, Fw);
}

// the end of the forward loop: the finiteness of z_T, and z_T to z_out [n][NZ] when it is wanted
template <int MODEL>
__device__ __forceinline__ void adj_fwd_end(const double* x, const double* Z, double* z_out, long long v, bool& bad) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) bad |= !adj_finite(x[q]);
#pragma unroll
    for (int q = 0; q < D::NL; ++q) bad |= D::THR && !adj_finite(Z[q]);
    if (z_out) {
#pragma unroll
        for (int q = 0; q < D::NX; ++q) z_out[v * D::NZ + q] = x[q];
        if constexpr (D::THR) {
#pragma unroll
            for (int q = 0; q < D::NL; ++q) z_out[v * D::NZ + D::NX + q] = Z[q];
        }
    }
}

// lam = dL/dx_T, mu = dL/dZ_T from gzT [n][NZ] (zero without it)
template <int MODEL>
__device__ __forceinline__ void adj_load_gzT(const double* gzT, long long v, double* lam, double* mu) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) lam[q] = gzT ? gzT[v * D::NZ + q] : 0.0;
#pragma unroll
    for (int q = 0; q < D::NL; ++q) mu[q] = (D::THR && gzT) ? gzT[v * D::NZ + D::NX + q] : 0.0;
}

// adds snapshot j of the trajectory cotangent gtraj [snapshots][n][NW]: NW = NX covers x (the rollout's snapshots),
// NW = NZ also the lag (the closed loop's)
template <int MODEL, int NW>
__device__ __forceinline__ void adj_add_gtraj(const double* gtraj, long long j, long long n, long long v, double* lam,
                                              double* mu) {
    using D = AdjDim<MODEL>;
    const double* gt = gtraj + (j * n + v) * NW;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) lam[q] += gt[q];
    if constexpr (D::THR && NW == D::NZ) {
#pragma unroll
        for (int q = 0; q < D::NL; ++q) mu[q] += gt[D::NX + q];
    }
}

// the step sizes of the reverse sweep, formed once before the loop
struct AdjDt {
    double dt, hdt, dt6, dt3;
};

// One reverse step: (lam, mu) = dL/d(x, Z)_{k+1} -> dL/d(x, Z)_k, and muF = dL/dFw_k.  x, Z: z_k (x is z_k again on
// return); Fw: the step's wrench; wk: z_k in the workspace.  It recomputes the stage states into sx, reverses the
// quaternion renormalisation and the lag (Z' = lagA Z_c + lagB Fw_c per channel), then sweeps the stages.  COEF: every
// stage also adds lambda^T df/dkp to the accumulator gk, with the current path always taken (nu - R^T 0 = nu), so
// gk[KP_CUR ..] exists without a current.  cur: the engine's has_current, read once at the top of the kernel (read
// here, it changes which products of rhs_quat13_vjp's rotation matrix the compiler fuses into fmas).
template <int MODEL, int INTEG, bool COEF, class P, class G = double*>
__device__ __forceinline__ void adj_step_vjp(const Consts<double>& c, const P& p, bool cur, const AdjDt& h, double* x,
                                             const double* Z, const double* Fw, const double* wk, long long n, double* sx,
                                             double* lam, double* mu, double* muF, const G& gk = G()) {
    using D = AdjDim<MODEL>;
    constexpr int NX = D::NX;
    constexpr bool THR = D::THR, QUAT = D::QUAT;
    // recompute the stage states (and the quaternion before its renormalisation)
    double qpre[4];
    if constexpr (INTEG == INTEG_RK4 || QUAT) {
        double xw[NX];
#pragma unroll
        for (int q = 0; q < NX; ++q) xw[q] = x[q];
        double acth;
        adj_step<MODEL, INTEG, true>(c, p, xw, Z, Fw, sx, qpre, acth);
    }
    if constexpr (QUAT) quat_normalize_vjp(qpre, lam + 3);
    if constexpr (THR) {
#pragma unroll
        for (int ch = 0; ch < 6; ++ch) {
            const double m0 = mu[3 * ch], m1 = mu[3 * ch + 1], m2 = mu[3 * ch + 2];
#pragma unroll
            for (int j = 0; j < 3; ++j) mu[3 * ch + j] = c.lagA[0][j] * m0 + c.lagA[1][j] * m1 + c.lagA[2][j] * m2;
            muF[ch] = c.lagB[0] * m0 + c.lagB[1] * m1 + c.lagB[2] * m2;
        }
    } else {
#pragma unroll
        for (int ch = 0; ch < 6; ++ch) muF[ch] = 0.0;
    }
    double lamp[NX], kap[NX];
#pragma unroll
    for (int q = 0; q < NX; ++q) lamp[q] = lam[q];
    // stage s at xs with the cotangent kap of its right-hand side: lam += a, the wrench cotangent b into
    // mu / muF (thruster: tau_s = lagG[s] . Z_c + lagH[s] Fw_c) or muF (wrench models: tau = u)
    auto stage_vjp = [&](int s, const double* xs, double* ga) {
        double b[6];
        if constexpr (COEF) {
            double tau[6];
            if constexpr (THR) {
                thruster_tau<double, true>(c, s, Z, Fw, tau);
            } else {
#pragma unroll
                for (int r = 0; r < 6; ++r) tau[r] = Fw[r];
            }
            if constexpr (QUAT) {
                rhs_quat13_vjp<true>(xs, p, true, kap, ga, b, tau, gk);
            } else {
                Trig<double> tr;
                trig_full<double>(c, xs + 3, tr);
                rhs_euler12_vjp<true>(xs, tr, p, true, kap, ga, b, tau, gk);
            }
        } else {
            if constexpr (QUAT) {
                rhs_quat13_vjp(xs, p, cur, kap, ga, b);
            } else {
                Trig<double> tr;
                trig_full<double>(c, xs + 3, tr);
                rhs_euler12_vjp(xs, tr, p, cur, kap, ga, b);
            }
        }
#pragma unroll
        for (int q = 0; q < NX; ++q) lam[q] += ga[q];
#pragma unroll
        for (int ch = 0; ch < 6; ++ch) {
            if constexpr (THR) {
#pragma unroll
                for (int j = 0; j < 3; ++j) mu[3 * ch + j] += c.lagG[s][j] * b[ch];
                muF[ch] += c.lagH[s] * b[ch];
            } else {
                muF[ch] += b[ch];
            }
        }
    };
    double ga[NX];
    if constexpr (INTEG == INTEG_EULER) {
#pragma unroll
        for (int q = 0; q < NX; ++q) kap[q] = h.dt * lamp[q];
        stage_vjp(0, x, ga);
    } else {
        // x' = x + dt/6 (k0 + 2 k1 + 2 k2 + k3), xs_s = x + h_s k_{s-1}
#pragma unroll
        for (int q = 0; q < NX; ++q) kap[q] = h.dt6 * lamp[q];
#pragma unroll
        for (int s = 3; s >= 1; --s) {
            double xs[NX];
#pragma unroll
            for (int q = 0; q < NX; ++q) xs[q] = sx[((s - 1) * NX + q) * ADJ_THREADS];
            stage_vjp(s, xs, ga);
            const double cs = (s == 1) ? h.dt6 : h.dt3;
            const double hs = (s == 3) ? h.dt : h.hdt;
#pragma unroll
            for (int q = 0; q < NX; ++q) kap[q] = fma(hs, ga[q], cs * lamp[q]);
        }
        // stage 0 is z_k itself: reloaded rather than held through the sweep (register pressure)
#pragma unroll
        for (int q = 0; q < NX; ++q) x[q] = wk[q * n];
        stage_vjp(0, x, ga);
    }
}

// dL/du_i from the wrench cotangent muF: thruster gu_i = F'(u_i) sum_c alloc[c][i] muF[c] (the allocation's
// structural zeros skipped, as in allocate_wrench); wrench models gu = muF
template <int MODEL>
__device__ __forceinline__ double adj_gu(const Consts<double>& c, const double* muF, const double* u, int i) {
    if constexpr (MODEL == MODEL_THRUSTER8) {
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const bool nz = (r < 2) ? (i < 4) : (r == 2) ? (i >= 4) : (r == 5) ? (i < 4) : true;
            if (nz) s += c.alloc[r][i] * muF[r];
        }
        return thrust_poly_d(c, u[i]) * s;
    } else {
        return muF[i];
    }
}

// (lam, mu) = dL/dz_0 to gz0 [n][NZ], with their finiteness
template <int MODEL>
__device__ __forceinline__ void adj_store_gz0(double* gz0, long long v, const double* lam, const double* mu, bool& bad) {
    using D = AdjDim<MODEL>;
#pragma unroll
    for (int q = 0; q < D::NX; ++q) {
        gz0[v * D::NZ + q] = lam[q];
        bad |= !adj_finite(lam[q]);
    }
    if constexpr (D::THR) {
#pragma unroll
        for (int q = 0; q < D::NL; ++q) {
            gz0[v * D::NZ + D::NX + q] = mu[q];
            bad |= !adj_finite(mu[q]);
        }
    }
}

// the block's counts of vehicles with a non-finite result (health[0]) and with a near-singular Euler step (health[1])
__device__ __forceinline__ void adj_health(unsigned long long* health, bool bad, bool sing) {
    if (health) {
        const int nb = __syncthreads_count(bad);
        const int ns = __syncthreads_count(sing);
        if (threadIdx.x == 0) {
            if (nb) atomicAdd(health + 0, (unsigned long long)nb);
            if (ns) atomicAdd(health + 1, (unsigned long long)ns);
        }
    }
}

// ---- the rollout sweeps (brov_rollout_vjp, brov_rollout_vjp_coef)

// vehicle v's sweep of an open-loop rollout: z_T to z_out, dL/du_k to gU, dL/dz_0 to gz0; COEF: lambda^T df/dkp of
// every stage into gk
template <int MODEL, int INTEG, bool COEF, class P, class G = double*>
__device__ __forceinline__ void adj_rollout_sweep(const AdjArgs& a, const P& p, bool cur, double* sx, long long v,
                                                  bool& bad, bool& sing, const G& gk = G()) {
    using D = AdjDim<MODEL>;
    constexpr int NX = D::NX, NU = D::NU, NZ = D::NZ, NL = D::NL;
    const Consts<double>& c = a.c;
    const long long n = a.n;
    // ---- forward: z_k -> workspace
    double x[NX], Z[NL];
    adj_load_z0<MODEL>(a.z0, v, x, Z);
    for (int k = 0; k < a.steps; ++k) {
        adj_store_z<MODEL>(a.ws + (long long)k * NZ * n + v, n, x, Z);
        adj_fwd_step<MODEL, INTEG>(c, p, x, Z, a.U + (long long)k * a.ust + v * a.usn, a.eps, sing);
    }
    adj_fwd_end<MODEL>(x, Z, a.z_out, v, bad);

    // ---- backward: lam = dL/dx_k, mu = dL/dZ_k
    double lam[NX], mu[NL];
    adj_load_gzT<MODEL>(a.gzT, v, lam, mu);
    if (a.gtraj && a.steps % a.stride == 0) adj_add_gtraj<MODEL, NX>(a.gtraj, a.steps / a.stride - 1, n, v, lam, mu);
    const double dt = c.dt, dt6 = dt * (1.0 / 6.0);
    const AdjDt h{dt, 0.5 * dt, dt6, 2.0 * dt6};
    for (int k = a.steps - 1; k >= 0; --k) {
        const double* wk = a.ws + (long long)k * NZ * n + v;
        adj_load_z<MODEL>(wk, n, x, Z);
        const double* uk = a.U + (long long)k * a.ust + v * a.usn;
        double Fw[6], muF[6];
        adj_wrench<MODEL>(c, uk, Fw);
        adj_step_vjp<MODEL, INTEG, COEF>(c, p, cur, h, x, Z, Fw, wk, n, sx, lam, mu, muF, gk);
        double* gu = a.gU + ((long long)k * n + v) * NU;
#pragma unroll
        for (int i = 0; i < NU; ++i) {
            const double g = adj_gu<MODEL>(c, muF, uk, i);
            gu[i] = g;
            bad |= !adj_finite(g);
        }
        if (a.gtraj && k > 0 && k % a.stride == 0) adj_add_gtraj<MODEL, NX>(a.gtraj, k / a.stride - 1, n, v, lam, mu);
    }
    adj_store_gz0<MODEL>(a.gz0, v, lam, mu, bad);
}

template <int MODEL, int INTEG>
__global__ void __launch_bounds__(ADJ_THREADS) adjoint_kernel(const __grid_constant__ AdjArgs a) {
    constexpr int NSTAGE = INTEG == INTEG_RK4 ? 3 * LinDim<MODEL>::NX * ADJ_THREADS : 1;
    __shared__ double stage[NSTAGE];      // RK4: [stage 1..3][i][thread], conflict-free
    const ParamsConst<double> p{a.c.kp};
    const bool cur = a.c.has_current != 0;
    const int tid = threadIdx.x;
    const long long v = (long long)blockIdx.x * ADJ_THREADS + tid;
    bool bad = false, sing = false;
    if (v < a.n) adj_rollout_sweep<MODEL, INTEG, false>(a, p, cur, stage + tid, v, bad, sing);
    adj_health(a.health, bad, sing);
}

// a shared-memory column of the coefficient cotangent: entry j of this thread at base[j * ADJ_THREADS]
struct CoefAcc {
    double* base;
    __device__ __forceinline__ double& operator[](int j) const { return base[j * ADJ_THREADS]; }
};

// adjoint_kernel's sweep with the coefficient cotangent (brov_rollout_vjp_coef): the thread's column gk of a
// shared-memory accumulator receives lambda^T df/dkp of every stage (rhs_*_vjp<true>, nu_dot_coef_vjp) in a fixed
// order and goes to gkp [KP_COUNT][n] at the end.  Dynamic shared memory, one column per thread (conflict-free):
// [RK4 stage buffer (3 NX) | gk (ADJ_NKPG) | PV: the vehicle's column of the per-vehicle table (KP_COUNT), staged as
// closed_loop_kernel stages it].
template <int MODEL, int INTEG, bool PV>
__global__ void __launch_bounds__(ADJ_THREADS) adjoint_coef_kernel(const __grid_constant__ AdjCoefArgs ca) {
    extern __shared__ double smem[];
    const AdjArgs& a = ca.a;
    const int tid = threadIdx.x;
    const long long v = (long long)blockIdx.x * ADJ_THREADS + tid;
    const long long n = a.n;
    double* col = smem + adj_stage_rows(MODEL, INTEG) * ADJ_THREADS + tid;
    const CoefAcc gk{col};
#pragma unroll
    for (int j = 0; j < ADJ_NKPG; ++j) gk[j] = 0.0;
    typename std::conditional<PV, ParamsShared<double>, ParamsConst<double>>::type p;
    if constexpr (PV) {
        const double* pvt = ca.pv + (v < n ? v : 0);
#pragma unroll 4
        for (int j = 0; j < KP_COUNT; ++j) col[(ADJ_NKPG + j) * ADJ_THREADS] = pvt[(long long)j * n];
        p.base = col + ADJ_NKPG * ADJ_THREADS;
        p.pitch = ADJ_THREADS;
    } else {
        p.kp = a.c.kp;
    }
    bool bad = false, sing = false;
    if (v < n) {
        adj_rollout_sweep<MODEL, INTEG, true>(a, p, true, smem + tid, v, bad, sing, gk);
#pragma unroll
        for (int j = 0; j < KP_COUNT; ++j) {
            const double g = j < ADJ_NKPG ? gk[j] : 0.0;
            ca.gkp[(long long)j * n + v] = g;
            bad |= !adj_finite(g);
        }
    }
    adj_health(a.health, bad, sing);
}


// ---------------------------------------------------------------------------------------------------------------
// closed-loop adjoint (brov_closed_loop_vjp)
// ---------------------------------------------------------------------------------------------------------------

// dz_j = z_j - zr_j, the Euler angles wrapped to one turn with closed_loop_kernel's arithmetic (derivative 1)
template <int MODEL>
__device__ __forceinline__ double cl_dz(double z, double zr, int j) {
    double d = z - zr;
    if (!ModelDim<MODEL>::QUAT && j >= 3 && j < 6) d = fma(-6.283185307179586, rint(d * 0.15915494309189535), d);
    return d;
}

// u = clamp(ur - K dz, u_min, u_max) with closed_loop_kernel's fixed-order fmas (per j, every channel); m[r]: channel r
// not clamped (a NaN takes that branch, as the compare-select does)
template <int MODEL>
__device__ __forceinline__ void cl_feedback(const ClAdjArgs& a, const double* __restrict__ x, const double* __restrict__ Z,
                                            const double* Kk, const double* zrk, const double* urk, double* __restrict__ u,
                                            bool* __restrict__ m) {
    constexpr int NX = LinDim<MODEL>::NX, NU = LinDim<MODEL>::NU, NZ = LinDim<MODEL>::NZ;
#pragma unroll
    for (int r = 0; r < NU; ++r) u[r] = __ldg(urk + r);
#pragma unroll
    for (int j = 0; j < NZ; ++j) {
        const double d = cl_dz<MODEL>(j < NX ? x[j] : Z[j < NX ? 0 : j - NX], __ldg(zrk + j), j);
#pragma unroll
        for (int r = 0; r < NU; ++r) u[r] = fma(-Kk[r * NZ + j], d, u[r]);
    }
#pragma unroll
    for (int r = 0; r < NU; ++r) {
        const bool lo = u[r] < a.u_min[r], hi = u[r] > a.u_max[r];
        m[r] = !(lo || hi);
        u[r] = lo ? a.u_min[r] : (hi ? a.u_max[r] : u[r]);
    }
}

// The sweep of brov_closed_loop_vjp: the rollout sweep's pieces with u_k from the feedback law.  Forward: z_k to the
// workspace, u_k, the primal step.  Reverse: reload z_k, recompute u_k (never stored), the step VJP (lambda_{k+1} ->
// A^T lambda, B^T lambda = adj_gu), then the feedback:
//     gv = m . (B^T lambda + 2 g_c r . (u - ur))          dL/dv_k, m the clamp mask
//     gdz = -K_k^T gv + 2 g_c q . dz_k                    lambda_k = A^T lambda + gdz + c_k (the lag rows into mu)
// and stores gv, dL/dur_k = gv - 2 g_c r . (u - ur) and dL/dzr_k = -gdz for the reductions.  Dynamic shared memory:
// [RK4 stage buffer (3 NX rows) | PV: the vehicle's table column (KP_COUNT rows) | the staged K (k_smem)].
template <int MODEL, int INTEG, bool PV>
__global__ void __launch_bounds__(ADJ_THREADS) closed_loop_adjoint_kernel(const __grid_constant__ ClAdjArgs a) {
    using D = AdjDim<MODEL>;
    constexpr int NX = D::NX, NU = D::NU, NZ = D::NZ, NL = D::NL;
    extern __shared__ double smem[];
    const Consts<double>& c = a.c;
    const bool cur = c.has_current != 0;
    const int tid = threadIdx.x;
    double* sx = smem + tid;
    const long long v = (long long)blockIdx.x * ADJ_THREADS + tid;
    const long long n = a.n;
    const long long vc = v < n ? v : n - 1;   // dead lanes stage the last vehicle's column, never store
    double* rest = smem + adj_stage_rows(MODEL, INTEG) * ADJ_THREADS;
    typename std::conditional<PV, ParamsShared<double>, ParamsConst<double>>::type p;
    if constexpr (PV) {
        const double* pvt = a.pv + vc;
#pragma unroll 4
        for (int j = 0; j < KP_COUNT; ++j) rest[j * ADJ_THREADS + tid] = pvt[(long long)j * n];
        p.base = rest + tid;
        p.pitch = ADJ_THREADS;
        rest += KP_COUNT * ADJ_THREADS;
    } else {
        p.kp = c.kp;
    }
    const double* Kp;
    if (a.k_smem) {
        for (int j = tid; j < NU * NZ; j += ADJ_THREADS) rest[j] = a.K[j];
        Kp = rest;
    } else {
        Kp = a.K + vc * a.K_sn;
    }
    __syncthreads();
    bool bad = false, sing = false;
    if (v < n) {
        const double* zrp = a.zr + v * a.zr_sn;
        const double* urp = a.ur + v * a.ur_sn;
        // ---- forward: z_k -> workspace
        double x[NX], Z[NL];
        adj_load_z0<MODEL>(a.z0, v, x, Z);
        for (int k = 0; k < a.steps; ++k) {
            adj_store_z<MODEL>(a.ws + (long long)k * NZ * n + v, n, x, Z);
            double u[NU];
            bool m[NU];
            cl_feedback<MODEL>(a, x, Z, Kp + (long long)k * a.K_st, zrp + (long long)k * a.zr_st,
                               urp + (long long)k * a.ur_st, u, m);
            adj_fwd_step<MODEL, INTEG>(c, p, x, Z, u, a.eps, sing);
        }
        adj_fwd_end<MODEL>(x, Z, a.z_out, v, bad);

        // ---- backward: lam = dL/dx_k, mu = dL/dZ_k
        double lam[NX], mu[NL];
        adj_load_gzT<MODEL>(a.gzT, v, lam, mu);
        if (a.gtraj && a.steps % a.stride == 0) adj_add_gtraj<MODEL, NZ>(a.gtraj, a.steps / a.stride - 1, n, v, lam, mu);
        const bool cost = a.gcost != nullptr;
        const double gc2 = cost ? 2.0 * a.gcost[v] : 0.0;
        const double dt = c.dt, dt6 = dt * (1.0 / 6.0);
        const AdjDt h{dt, 0.5 * dt, dt6, 2.0 * dt6};
        for (int k = a.steps - 1; k >= 0; --k) {
            const double* wk = a.ws + (long long)k * NZ * n + v;
            adj_load_z<MODEL>(wk, n, x, Z);
            const double* Kk = Kp + (long long)k * a.K_st;
            const double* zrk = zrp + (long long)k * a.zr_st;
            const double* urk = urp + (long long)k * a.ur_st;
            double u[NU];
            bool m[NU];
            cl_feedback<MODEL>(a, x, Z, Kk, zrk, urk, u, m);
            double Fw[6], muF[6];
            adj_wrench<MODEL>(c, u, Fw);
            adj_step_vjp<MODEL, INTEG, false>(c, p, cur, h, x, Z, Fw, wk, n, sx, lam, mu, muF);
            // the feedback: gv and dL/dur from gu = B^T lambda
            double gv[NU];
#pragma unroll
            for (int i = 0; i < NU; ++i) {
                const double g = adj_gu<MODEL>(c, muF, u, i);
                const double gc = cost ? gc2 * a.r[i] * (u[i] - __ldg(urk + i)) : 0.0;
                gv[i] = m[i] ? g + gc : 0.0;
                const double gur = gv[i] - gc;
                bad |= !adj_finite(gur);
                if (a.wgv) a.wgv[((long long)k * NU + i) * n + v] = gv[i];
                if (a.wgur) a.wgur[((long long)k * NU + i) * n + v] = gur;
            }
            // lambda_k = A^T lambda + gdz (+ c_k below); dL/dzr_k = -gdz.  With the gain gradient requested, its entries
            // -gv_r dz_j are all finite exactly when max_r |gv_r| max_j |dz_j| is (the dz maximum keeps a NaN; a
            // non-finite gv is counted through dL/dur)
            const bool gk = a.wgv != nullptr;
            double dmax = 0.0;
#pragma unroll
            for (int j = 0; j < NZ; ++j) {
                const double zj = j < NX ? x[j] : Z[j < NX ? 0 : j - NX];
                const double d = (cost || gk) ? cl_dz<MODEL>(zj, __ldg(zrk + j), j) : 0.0;
                dmax = fabs(d) > dmax || d != d ? fabs(d) : dmax;
                double g = cost ? gc2 * a.q[j] * d : 0.0;
#pragma unroll
                for (int r = 0; r < NU; ++r) g = fma(-Kk[r * NZ + j], gv[r], g);
                if (j < NX) lam[j] += g; else mu[j < NX ? 0 : j - NX] += g;
                bad |= !adj_finite(g);
                if (a.wgzr) a.wgzr[((long long)k * NZ + j) * n + v] = -g;
            }
            if (gk) {
                double gvmax = 0.0;
#pragma unroll
                for (int r = 0; r < NU; ++r) gvmax = fabs(gv[r]) > gvmax ? fabs(gv[r]) : gvmax;
                bad |= !adj_finite(gvmax * dmax);
            }
            if (a.gtraj && k > 0 && k % a.stride == 0) adj_add_gtraj<MODEL, NZ>(a.gtraj, k / a.stride - 1, n, v, lam, mu);
        }
        adj_store_gz0<MODEL>(a.gz0, v, lam, mu, bad);
    }
    adj_health(a.health, bad, sing);
}

// ---- the launches: one model x integrator (x PV) ladder

template <int V> using AdjInt = std::integral_constant<int, V>;
template <bool V> using AdjBool = std::integral_constant<bool, V>;

// go(model, integ, pv) with compile-time tags; PV only where pv is set
template <class Go>
static cudaError_t adj_dispatch(int model, int integ, bool pv, Go go) {
    auto by_integ = [&](auto m) -> cudaError_t {
        if (integ == INTEG_RK4) return pv ? go(m, AdjInt<INTEG_RK4>(), AdjBool<true>()) : go(m, AdjInt<INTEG_RK4>(), AdjBool<false>());
        return pv ? go(m, AdjInt<INTEG_EULER>(), AdjBool<true>()) : go(m, AdjInt<INTEG_EULER>(), AdjBool<false>());
    };
    switch (model) {
        case MODEL_THRUSTER8: return by_integ(AdjInt<MODEL_THRUSTER8>());
        case MODEL_WRENCH12: return by_integ(AdjInt<MODEL_WRENCH12>());
        case MODEL_QUAT13: return by_integ(AdjInt<MODEL_QUAT13>());
    }
    return cudaErrorInvalidValue;
}

// one thread per vehicle in blocks of ADJ_THREADS, with smem bytes of dynamic shared memory
template <class Args>
static cudaError_t adj_launch(void (*kern)(Args), size_t smem, long long n, const Args& a, cudaStream_t st) {
    if (smem) {
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long long grid = (n + ADJ_THREADS - 1) / ADJ_THREADS;
    kern<<<(unsigned)grid, ADJ_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_adjoint(int model, int integ, const AdjArgs& a, cudaStream_t st) {
    return adj_dispatch(model, integ, false, [&](auto m, auto i, auto) {
        return adj_launch(adjoint_kernel<decltype(m)::value, decltype(i)::value>, 0, a.n, a, st);
    });
}

cudaError_t launch_adjoint_coef(int model, int integ, const AdjCoefArgs& a, cudaStream_t st) {
    return adj_dispatch(model, integ, a.pv != nullptr, [&](auto m, auto i, auto pv) {
        constexpr int M = decltype(m)::value, I = decltype(i)::value;
        constexpr bool PV = decltype(pv)::value;
        return adj_launch(adjoint_coef_kernel<M, I, PV>, adj_smem_bytes(M, I, ADJ_NKPG + (PV ? KP_COUNT : 0), 0), a.a.n, a, st);
    });
}

cudaError_t launch_closed_loop_adjoint(int model, int integ, const ClAdjArgs& a, cudaStream_t st) {
    return adj_dispatch(model, integ, a.pv != nullptr, [&](auto m, auto i, auto pv) {
        constexpr int M = decltype(m)::value, I = decltype(i)::value;
        constexpr bool PV = decltype(pv)::value;
        const size_t k_bytes = a.k_smem ? (size_t)LinDim<M>::NU * LinDim<M>::NZ * sizeof(double) : 0;
        return adj_launch(closed_loop_adjoint_kernel<M, I, PV>, adj_smem_bytes(M, I, PV ? KP_COUNT : 0, k_bytes), a.n, a, st);
    });
}

// ---- the operand gradients: per (step k, vehicle i) Y rows of R values; value r of row y is element elem(y, r)
struct ClRedArgs {
    const double* ws;             // z_k [steps][NZ][n]
    const double* wgv;            // [steps][NU][n]
    const double* src;            // WHICH 1 / 2: [steps][Y][n]; SCR: the scratch [E][n] (one "step")
    const double* zr;
    long long zr_st, zr_sn;
    double* out;                  // element (k, i, e) at out[k*st + i*sn + e*se]
    long long st, sn, se;
    long long n;
    int steps;
};

template <int MODEL, int WHICH, bool SCR> struct ClRed {
    static constexpr int NZ = LinDim<MODEL>::NZ, NU = LinDim<MODEL>::NU;
    static constexpr int E = WHICH == 0 ? NU * NZ : (WHICH == 1 ? NZ : NU);   // elements of the operand
    static constexpr int Y = SCR ? E : (WHICH == 2 ? NU : NZ);
    static constexpr int R = (WHICH == 0 && !SCR) ? NU : 1;
    static __device__ __forceinline__ long long elem(int y, int r) { return R > 1 ? (long long)r * NZ + y : y; }
    static __device__ __forceinline__ void load(const ClRedArgs& a, long long k, long long i, int y, double* val) {
        const long long n = a.n;
        if constexpr (R > 1) {
            // dL/dK_k = -gv dz^T
            const double d = cl_dz<MODEL>(a.ws[(k * NZ + y) * n + i], a.zr[k * a.zr_st + i * a.zr_sn + y], y);
#pragma unroll
            for (int r = 0; r < R; ++r) val[r] = -(a.wgv[(k * NU + r) * n + i] * d);
        } else {
            val[0] = a.src[(k * Y + y) * n + i];
        }
    }
};

// one thread per (vehicle, row), 32 vehicles x Y rows per block.  TNC: every (step, vehicle) has its own elements, the
// steps spread over gridDim.y; otherwise the sum over the steps in order k = 0, 1, ... (a per-vehicle operand, or the
// first stage of a shared constant one)
template <int MODEL, int WHICH, bool TNC>
__global__ void __launch_bounds__(1024) cl_red_steps_kernel(const ClRedArgs a) {
    using S = ClRed<MODEL, WHICH, false>;
    const long long i = (long long)blockIdx.x * 32 + threadIdx.x;
    const int y = threadIdx.y;
    if (i >= a.n) return;
    double val[S::R];
    if constexpr (TNC) {
        for (long long k = blockIdx.y; k < a.steps; k += gridDim.y) {
            S::load(a, k, i, y, val);
#pragma unroll
            for (int r = 0; r < S::R; ++r) a.out[k * a.st + i * a.sn + S::elem(y, r) * a.se] = val[r];
        }
    } else {
        double acc[S::R];
#pragma unroll
        for (int r = 0; r < S::R; ++r) acc[r] = 0.0;
        for (long long k = 0; k < a.steps; ++k) {
            S::load(a, k, i, y, val);
#pragma unroll
            for (int r = 0; r < S::R; ++r) acc[r] += val[r];
        }
#pragma unroll
        for (int r = 0; r < S::R; ++r) a.out[i * a.sn + S::elem(y, r) * a.se] = acc[r];
    }
}

// the sum over the vehicles of row (k, y), one block per row: thread t adds vehicles t, t + 256, ... in order, then a
// fixed shared-memory tree over the threads
constexpr int CL_RED_THREADS = 256;
template <int MODEL, int WHICH, bool SCR>
__global__ void __launch_bounds__(CL_RED_THREADS) cl_red_vehicles_kernel(const ClRedArgs a) {
    using S = ClRed<MODEL, WHICH, SCR>;
    __shared__ double red[S::R][CL_RED_THREADS];
    const int t = threadIdx.x;
    const long long rows = (long long)a.steps * S::Y;
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const long long k = row / S::Y;
        const int y = (int)(row % S::Y);
        double acc[S::R], val[S::R];
#pragma unroll
        for (int r = 0; r < S::R; ++r) acc[r] = 0.0;
        for (long long i = t; i < a.n; i += CL_RED_THREADS) {
            S::load(a, k, i, y, val);
#pragma unroll
            for (int r = 0; r < S::R; ++r) acc[r] += val[r];
        }
#pragma unroll
        for (int r = 0; r < S::R; ++r) red[r][t] = acc[r];
        __syncthreads();
        for (int h = CL_RED_THREADS / 2; h > 0; h >>= 1) {
            if (t < h) {
#pragma unroll
                for (int r = 0; r < S::R; ++r) red[r][t] += red[r][t + h];
            }
            __syncthreads();
        }
        if (t < S::R) a.out[k * a.st + S::elem(y, t) * a.se] = red[t][0];
        __syncthreads();
    }
}

template <int MODEL, int WHICH>
static cudaError_t cl_reduce(const ClAdjArgs& c, double* out, long long st, long long sn, double* scratch, cudaStream_t s) {
    using S = ClRed<MODEL, WHICH, false>;
    ClRedArgs a;
    a.ws = c.ws;
    a.wgv = c.wgv;
    a.src = WHICH == 1 ? c.wgzr : c.wgur;
    a.zr = c.zr; a.zr_st = c.zr_st; a.zr_sn = c.zr_sn;
    a.out = out; a.st = st; a.sn = sn; a.se = 1;
    a.n = c.n;
    a.steps = c.steps;
    const dim3 blk(32, S::Y);
    const unsigned gx = (unsigned)((c.n + 31) / 32);
    const unsigned vgrid = (unsigned)std::min<long long>((long long)c.steps * S::Y, 1LL << 20);
    if (st != 0 && sn != 0) {
        cl_red_steps_kernel<MODEL, WHICH, true><<<dim3(gx, (unsigned)std::min(c.steps, 65535)), blk, 0, s>>>(a);
    } else if (sn != 0) {
        cl_red_steps_kernel<MODEL, WHICH, false><<<gx, blk, 0, s>>>(a);
    } else if (st != 0) {
        cl_red_vehicles_kernel<MODEL, WHICH, false><<<vgrid, CL_RED_THREADS, 0, s>>>(a);
    } else {
        // shared and constant: the per-vehicle sums over the steps into scratch [E][n], then their sum over vehicles
        ClRedArgs b = a;
        b.out = scratch; b.st = 0; b.sn = 1; b.se = c.n;
        cl_red_steps_kernel<MODEL, WHICH, false><<<gx, blk, 0, s>>>(b);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        b = a;
        b.src = scratch;
        b.steps = 1;
        cl_red_vehicles_kernel<MODEL, WHICH, true><<<ClRed<MODEL, WHICH, true>::Y, CL_RED_THREADS, 0, s>>>(b);
    }
    return cudaGetLastError();
}

template <int MODEL>
static cudaError_t cl_reduce_which(int which, const ClAdjArgs& a, double* out, long long st, long long sn, double* scr,
                                   cudaStream_t s) {
    switch (which) {
        case 0: return cl_reduce<MODEL, 0>(a, out, st, sn, scr, s);
        case 1: return cl_reduce<MODEL, 1>(a, out, st, sn, scr, s);
        case 2: return cl_reduce<MODEL, 2>(a, out, st, sn, scr, s);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_closed_loop_adjoint_reduce(int model, int which, const ClAdjArgs& a, double* out, long long st,
                                              long long sn, double* scratch, cudaStream_t s) {
    if (a.n <= 0 || a.steps <= 0) return cudaSuccess;
    switch (model) {
        case MODEL_THRUSTER8: return cl_reduce_which<MODEL_THRUSTER8>(which, a, out, st, sn, scratch, s);
        case MODEL_WRENCH12: return cl_reduce_which<MODEL_WRENCH12>(which, a, out, st, sn, scratch, s);
        case MODEL_QUAT13: return cl_reduce_which<MODEL_QUAT13>(which, a, out, st, sn, scratch, s);
    }
    return cudaErrorInvalidValue;
}

}  // namespace brov
