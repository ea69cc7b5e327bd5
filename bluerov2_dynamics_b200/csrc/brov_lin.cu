// brov_lin.cu — exact Jacobians of the discrete step, A_k = dPhi/dz (z_k, u_k) and B_k = dPhi/du (z_k, u_k), along
// batched trajectories.
//
//   linearize_kernel   one thread per (vehicle, column j of J = [A | B]).  At every step the thread seeds the tangent of
//                      its column (x.d = e_j for a state column; the body wrench's tangent for a lag or input column),
//                      takes one dual step from the primal (z_k, u_k), writes column j of J_k and continues with the
//                      primal z_{k+1}.  The primal is recomputed by every thread of a vehicle (identical arithmetic,
//                      identical bits), as se_grad_kernel does per direction, so no thread waits on another inside a
//                      step.  A block stages the J_k of its V vehicles in shared memory and writes it out contiguously.
//
// The thruster map and the lag stay outside the dual arithmetic: within a step the lag is a fixed linear filter of the
// held input, so the wrench's tangent at sub-step s is a per-thread constant and the lag rows of J are closed form.
// The coefficients carry no tangent: the right-hand side reads them as plain doubles (ParamsConst).
#include "brov_lin.cuh"

namespace brov {

// a tangent-free operand: no zero tangent to add (ptxas cannot fold x + 0.0)
__device__ __forceinline__ Dual operator+(Dual a, double b) { return Dual(a.v + b, a.d); }
__device__ __forceinline__ Dual operator-(Dual a, double b) { return Dual(a.v - b, a.d); }

// One integrator step with the state as dual numbers.  The body wrench of sub-step s has the value of Fw (thruster: the
// allocated static thrust, turned into the lagged wrench here; wrench models: the input) and the tangent g_s * tvec,
// g_s = lagG[s][lagk] for a lag column and lagH[s] otherwise (thruster), 1 (wrench models).  Same stage structure as
// integrate_step_dual, every stage with full sines and cosines; the lag is not advanced here.
template <int MODEL, int INTEG>
__device__ __forceinline__ void integrate_step_lin(const Consts<double>& c, Dual* __restrict__ x,
                                                   const double* __restrict__ lag, const double* __restrict__ Fw,
                                                   const double* __restrict__ tvec, int lagk, double& abs_cth) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr bool EULER_ANGLES = !ModelDim<MODEL>::QUAT;
    const ParamsConst<double> p{c.kp};
    const bool cur = c.has_current != 0;
    const double dt = c.dt;
    auto rhs = [&](int s, const Dual* xs, Dual* out) {
        Dual tau[6];
        if constexpr (MODEL == MODEL_THRUSTER8) {
            double t[6];
            thruster_tau<double, true>(c, s, lag, Fw, t);
            // lag column (c, k): lagG[s][k] in row c; input column i: lagH[s] alloc[:, i] F'(u_i); state column: 0
            const double g = lagk == 0 ? c.lagG[s][0] : lagk == 1 ? c.lagG[s][1] : lagk == 2 ? c.lagG[s][2] : c.lagH[s];
#pragma unroll
            for (int r = 0; r < 6; ++r) tau[r] = Dual(t[r], g * tvec[r]);
        } else {
#pragma unroll
            for (int r = 0; r < 6; ++r) tau[r] = Dual(Fw[r], tvec[r]);
        }
        if constexpr (EULER_ANGLES) {
            Trig<Dual> tr;
            trig_full<Dual>(xs + 3, tr);
            if (s == 0) abs_cth = fabs(tr.cth.v);
            rhs_euler12<Dual>(xs, tr, tau, p, cur, out);
        } else {
            rhs_quat13<Dual>(xs, tau, p, cur, out);
        }
    };
    if constexpr (!EULER_ANGLES) abs_cth = 1.0;
    Dual k[NX];
    if constexpr (INTEG == INTEG_EULER) {
        rhs(0, x, k);
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt * k[i];
    } else {
        Dual acc[NX], xs[NX];
        const double hdt = 0.5 * dt;
        rhs(0, x, k);
#pragma unroll
        for (int s = 1; s <= 3; ++s) {
            const double w = (s == 1) ? 1.0 : 2.0;
            const double h = (s == 3) ? dt : hdt;
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                if (s == 1) acc[i] = k[i]; else acc[i] += w * k[i];
                xs[i] = x[i] + h * k[i];
            }
            rhs(s, xs, k);
        }
        const double dt6 = dt * (1.0 / 6.0);
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt6 * (acc[i] + k[i]);
    }
    if constexpr (ModelDim<MODEL>::QUAT) quat_renorm<Dual>(x + 3);
}

__device__ __forceinline__ bool finite_(double v) { return fabs(v) <= 1.7976931348623157e308; }

template <int MODEL, int INTEG>
__global__ void __launch_bounds__(LinDim<MODEL>::THREADS) linearize_kernel(const __grid_constant__ LinArgs a) {
    using D = LinDim<MODEL>;
    constexpr int NX = D::NX, NU = D::NU, NZ = D::NZ, NC = D::NC, V = D::V;
    constexpr bool THR = MODEL == MODEL_THRUSTER8;
    constexpr int NL = THR ? 18 : 1;
    constexpr int TILE = V * NZ * NC;
    __shared__ double tile[TILE];          // [V][NZ][NC]: J_k of the block's vehicles, as laid out in memory
    __shared__ int flags[V];               // bit 0: non-finite result, bit 1: came near theta = +-pi/2
    const int tid = threadIdx.x;
    const int vl = tid / NC, j = tid - vl * NC;
    const long long v0 = (long long)blockIdx.x * V;
    const long long v = v0 + vl;
    const bool act = v < a.n;
    const int nv = (int)(a.n - v0 < V ? a.n - v0 : V);
    if (tid < V) flags[tid] = 0;
    double x[NX], lag[NL];
#pragma unroll
    for (int q = 0; q < NX; ++q) x[q] = act ? a.z0[v * NZ + q] : 0.0;
#pragma unroll
    for (int q = 0; q < NL; ++q) lag[q] = (THR && act) ? a.z0[v * NZ + NX + q] : 0.0;
    // column kind: state j < NX, lag column (lc, lagk) for NX <= j < NZ, input column ui = j - NZ
    const int ui = j - NZ;
    const int lj = j - NX;
    const int lc = (THR && lj >= 0 && ui < 0) ? lj / 3 : -1;
    const int lagk = lc >= 0 ? lj - 3 * lc : -1;
    bool bad = false, sing = false;
    for (int k = 0; k < a.steps; ++k) {
        if (act) {
            const double* uk = a.U + (long long)k * a.ust + v * a.usn;
            double u[NU];
#pragma unroll
            for (int q = 0; q < NU; ++q) u[q] = uk[q];
            double Fw[6], tvec[6];
            if constexpr (THR) {
                double F[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) F[i] = thrust_poly<double>(a.c, u[i]);
                allocate_wrench<double>(a.c, F, Fw);
                // input column: alloc[:, ui] F'(u_ui); lag column: e_lc; state column: 0
                const double fp = ui >= 0 ? thrust_poly_d(a.c, uk[ui]) : 0.0;
#pragma unroll
                for (int r = 0; r < 6; ++r) tvec[r] = ui >= 0 ? a.c.alloc[r][ui] * fp : (r == lc ? 1.0 : 0.0);
            } else {
#pragma unroll
                for (int r = 0; r < 6; ++r) { Fw[r] = u[r]; tvec[r] = r == ui ? 1.0 : 0.0; }
            }
            Dual xd[NX];
#pragma unroll
            for (int q = 0; q < NX; ++q) xd[q] = Dual(x[q], q == j ? 1.0 : 0.0);
            double acth;
            integrate_step_lin<MODEL, INTEG>(a.c, xd, lag, Fw, tvec, lagk, acth);
            sing |= acth < a.eps;
            double* col = tile + vl * NZ * NC + j;
#pragma unroll
            for (int q = 0; q < NX; ++q) {
                col[q * NC] = xd[q].d;
                bad |= !finite_(xd[q].d);
                x[q] = xd[q].v;
            }
            if constexpr (THR) {
                // dZ'/dx = 0, dZ'/dZ = lagA per channel, dZ'/du_i = lagB (x) alloc[:, i] F'(u_i)
#pragma unroll
                for (int cc = 0; cc < 6; ++cc) {
#pragma unroll
                    for (int kk = 0; kk < 3; ++kk) {
                        double jv = 0.0;
                        if (ui >= 0) jv = a.c.lagB[kk] * tvec[cc];
                        else if (cc == lc) jv = lagk == 0 ? a.c.lagA[kk][0] : lagk == 1 ? a.c.lagA[kk][1] : a.c.lagA[kk][2];
                        col[(NX + 3 * cc + kk) * NC] = jv;
                        bad |= !finite_(jv);
                    }
                }
                lag_advance<double, true>(a.c, lag, Fw);
            }
            if (j == 0) {
#pragma unroll
                for (int q = 0; q < NX; ++q) bad |= !finite_(x[q]);
#pragma unroll
                for (int q = 0; q < NL; ++q) bad |= THR && !finite_(lag[q]);
                if (a.z_traj) {
                    double* zt = a.z_traj + ((long long)k * a.n + v) * NZ;
#pragma unroll
                    for (int q = 0; q < NX; ++q) zt[q] = x[q];
                    if constexpr (THR) {
#pragma unroll
                        for (int q = 0; q < NL; ++q) zt[NX + q] = lag[q];
                    }
                }
            }
        }
        __syncthreads();
        double* out = a.jac + ((long long)k * a.n + v0) * (NZ * NC);
        for (int e = tid; e < nv * NZ * NC; e += D::THREADS) out[e] = tile[e];
        __syncthreads();
    }
    if (act && j == 0 && a.z_out) {
#pragma unroll
        for (int q = 0; q < NX; ++q) a.z_out[v * NZ + q] = x[q];
        if constexpr (THR) {
#pragma unroll
            for (int q = 0; q < NL; ++q) a.z_out[v * NZ + NX + q] = lag[q];
        }
    }
    if (a.health) {
        if (act && (bad || sing)) atomicOr(&flags[vl], (bad ? 1 : 0) | (sing && j == 0 ? 2 : 0));
        __syncthreads();
        if (tid == 0) {
            unsigned long long nb = 0, ns = 0;
            for (int w = 0; w < nv; ++w) { nb += flags[w] & 1; ns += (flags[w] >> 1) & 1; }
            if (nb) atomicAdd(a.health + 0, nb);
            if (ns) atomicAdd(a.health + 1, ns);
        }
    }
}

template <int MODEL, int INTEG>
static cudaError_t linearize_go(const LinArgs& a, cudaStream_t st) {
    using D = LinDim<MODEL>;
    const long long grid = (a.n + D::V - 1) / D::V;
    linearize_kernel<MODEL, INTEG><<<(unsigned)grid, D::THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

template <int MODEL>
static cudaError_t linearize_integ(int integ, const LinArgs& a, cudaStream_t st) {
    return integ == INTEG_RK4 ? linearize_go<MODEL, INTEG_RK4>(a, st) : linearize_go<MODEL, INTEG_EULER>(a, st);
}

cudaError_t launch_linearize(int model, int integ, const LinArgs& a, cudaStream_t st) {
    switch (model) {
        case MODEL_THRUSTER8: return linearize_integ<MODEL_THRUSTER8>(integ, a, st);
        case MODEL_WRENCH12: return linearize_integ<MODEL_WRENCH12>(integ, a, st);
        case MODEL_QUAT13: return linearize_integ<MODEL_QUAT13>(integ, a, st);
    }
    return cudaErrorInvalidValue;
}

// ekf_kernel   one thread per (filter, state column j), NX threads per filter.  At every step thread j takes the dual
//              step seeded along e_j (the primal is recomputed identically by every thread of the filter, as in
//              linearize_kernel) and writes column j of A_k into shared memory.  Thread i then forms row i of A P and
//              the upper triangle of row i of A P A^T + diag(q), mirrored, so P stays exactly symmetric.  The scalar
//              updates run over the measured components in order; each writes the Joseph-form P into the other half
//              of a per-filter ping-pong buffer.  Every thread of a block executes the same barrier sequence: a filter
//              with nothing measured at component m skips the arithmetic, not the barrier.
template <int MODEL, int INTEG>
__global__ void __launch_bounds__(EkfDim<MODEL>::THREADS) ekf_kernel(const __grid_constant__ EkfArgs a) {
    using D = EkfDim<MODEL>;
    constexpr int NX = D::NX, NU = D::NU, NZ = D::NZ, V = D::V, NN = NX * NX;
    constexpr bool THR = MODEL == MODEL_THRUSTER8;
    constexpr int NL = THR ? 18 : 1;
    constexpr double TWO_PI = 6.283185307179586, INV_2PI = 0.15915494309189535, LOG_2PI = 1.8378770664093453;
    __shared__ double sA[V * NN];          // [V][NX][NX]: A_k of the block's filters
    __shared__ double sP[2 * V * NN];      // [2][V][NX][NX]: P and the temporary, swapped by the updates
    __shared__ int flags[V];               // bit 0: non-finite result, bit 1: came near theta = +-pi/2
    const int tid = threadIdx.x;
    const int fl = tid / NX, j = tid - fl * NX;
    const long long f = (long long)blockIdx.x * V + fl;
    const bool act = f < a.n;
    const int nv = (int)(a.n - (long long)blockIdx.x * V < V ? a.n - (long long)blockIdx.x * V : V);
    if (tid < V) flags[tid] = 0;
    double* A = sA + fl * NN;
    int cur = 0;                           // which half of sP holds this filter's P (the same in all its threads)
    double x[NX], lag[NL];
#pragma unroll
    for (int q = 0; q < NX; ++q) x[q] = act ? a.z0[f * NZ + q] : 0.0;
#pragma unroll
    for (int q = 0; q < NL; ++q) lag[q] = (THR && act) ? a.z0[f * NZ + NX + q] : 0.0;
    if (act) {
#pragma unroll
        for (int c = 0; c < NX; ++c) sP[fl * NN + j * NX + c] = a.P0[f * NN + j * NX + c];
    }
    const double qj = act ? a.q[f * a.qsn + j] : 0.0;
    const double* rf = a.r + (act ? f : 0) * a.rsn;
    double ll = 0.0, nis = 0.0;
    long long cnt = 0;
    if (a.loglik && a.accumulate && act) { ll = a.loglik[f]; nis = a.nis[f]; cnt = a.count[f]; }
    bool sing = false;
    int countdown = a.stride;
    long long snap = 0;
    const double zero6[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int k = 0; k < a.steps; ++k) {
        // predict: the primal step and column j of A_k
        if (act) {
            const double* uk = a.U + (long long)k * a.ust + f * a.usn;
            double Fw[6];
            if constexpr (THR) {
                double F[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) F[i] = thrust_poly<double>(a.c, uk[i]);
                allocate_wrench<double>(a.c, F, Fw);
            } else {
#pragma unroll
                for (int r = 0; r < NU; ++r) Fw[r] = uk[r];
            }
            Dual xd[NX];
#pragma unroll
            for (int q = 0; q < NX; ++q) xd[q] = Dual(x[q], q == j ? 1.0 : 0.0);
            double acth;
            integrate_step_lin<MODEL, INTEG>(a.c, xd, lag, Fw, zero6, -1, acth);
            sing |= acth < a.eps;
#pragma unroll
            for (int q = 0; q < NX; ++q) {
                A[q * NX + j] = xd[q].d;
                x[q] = xd[q].v;
            }
            if constexpr (THR) lag_advance<double, true>(a.c, lag, Fw);
        }
        __syncthreads();
        if (act) {   // row j of A P into the free half
            const double* P = sP + cur * V * NN + fl * NN;
            double* Tm = sP + (cur ^ 1) * V * NN + fl * NN;
#pragma unroll
            for (int c = 0; c < NX; ++c) {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < NX; ++q) s = fma(A[j * NX + q], P[q * NX + c], s);
                Tm[j * NX + c] = s;
            }
        }
        __syncthreads();
        if (act) {   // row j of (A P) A^T + diag(q), upper triangle, mirrored
            double* P = sP + cur * V * NN + fl * NN;
            const double* Tm = sP + (cur ^ 1) * V * NN + fl * NN;
#pragma unroll
            for (int c = 0; c < NX; ++c) {
                if (c < j) continue;
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < NX; ++q) s = fma(Tm[j * NX + q], A[c * NX + q], s);
                if (c == j) s += qj;
                P[j * NX + c] = s;
                P[c * NX + j] = s;
            }
        }
        __syncthreads();
        // update: one scalar measurement per component, in order
        const double* yk = a.Y + (long long)k * a.yst + f * a.ysn;
#pragma unroll
        for (int m = 0; m < NX; ++m) {
            const double y = act ? yk[m] : 0.0;
            if (act && finite_(y)) {
                const double* P = sP + cur * V * NN + fl * NN;
                double* Pn = sP + (cur ^ 1) * V * NN + fl * NN;
                const double rm = rf[m];
                double nu = y - x[m];
                if (m >= 3 && m < 6) nu = fma(-TWO_PI, rint(nu * INV_2PI), nu);
                const double pmm = P[m * NX + m];
                const double s = pmm + rm;
                const double inv_s = 1.0 / s;   // one division per update: g = P[:, m] (1 / s)
                double g[NX];
#pragma unroll
                for (int c = 0; c < NX; ++c) {
                    g[c] = P[m * NX + c] * inv_s;
                    x[c] = fma(g[c], nu, x[c]);
                }
                // Joseph form: (I - g e_m^T) P (I - g e_m^T)^T + r g g^T, entry (j, c)
                const double gj = P[m * NX + j] * inv_s;
                const double kjm = P[j * NX + m] - gj * pmm;
#pragma unroll
                for (int c = 0; c < NX; ++c) {
                    if (c < j) continue;
                    const double v = (P[j * NX + c] - gj * P[m * NX + c]) - kjm * g[c] + rm * gj * g[c];
                    Pn[j * NX + c] = v;
                    Pn[c * NX + j] = v;
                }
                const double e2 = nu * nu * inv_s;
                ll -= 0.5 * (e2 + log(s) + LOG_2PI);
                nis += e2;
                ++cnt;
                cur ^= 1;
            }
            __syncthreads();
        }
        if (--countdown == 0) {
            countdown = a.stride;
            if (act) {
                const double* P = sP + cur * V * NN + fl * NN;
                if (a.x_traj) {
                    double xj = x[0];   // x[j] without a dynamically indexed (local-memory) array
#pragma unroll
                    for (int q = 1; q < NX; ++q) xj = q == j ? x[q] : xj;
                    a.x_traj[(snap * a.n + f) * NX + j] = xj;
                }
                if (a.P_traj) {
                    double* pt = a.P_traj + ((snap * a.n + f) * NX + j) * NX;
#pragma unroll
                    for (int c = 0; c < NX; ++c) pt[c] = P[j * NX + c];
                }
            }
            ++snap;
        }
    }
    bool bad = false;
    if (act) {
        const double* P = sP + cur * V * NN + fl * NN;
#pragma unroll
        for (int c = 0; c < NX; ++c) {
            a.P_out[f * NN + j * NX + c] = P[j * NX + c];
            bad |= !finite_(P[j * NX + c]);
        }
        if (j == 0) {
#pragma unroll
            for (int q = 0; q < NX; ++q) {
                a.z_out[f * NZ + q] = x[q];
                bad |= !finite_(x[q]);
            }
            if constexpr (THR) {
#pragma unroll
                for (int q = 0; q < NL; ++q) {
                    a.z_out[f * NZ + NX + q] = lag[q];
                    bad |= !finite_(lag[q]);
                }
            }
            if (a.loglik) { a.loglik[f] = ll; a.nis[f] = nis; a.count[f] = cnt; }
        }
    }
    if (a.health) {
        if (act && (bad || sing)) atomicOr(&flags[fl], (bad ? 1 : 0) | (sing && j == 0 ? 2 : 0));
        __syncthreads();
        if (tid == 0) {
            unsigned long long nb = 0, ns = 0;
            for (int w = 0; w < nv; ++w) { nb += flags[w] & 1; ns += (flags[w] >> 1) & 1; }
            if (nb) atomicAdd(a.health + 0, nb);
            if (ns) atomicAdd(a.health + 1, ns);
        }
    }
}

template <int MODEL, int INTEG>
static cudaError_t ekf_go(const EkfArgs& a, cudaStream_t st) {
    using D = EkfDim<MODEL>;
    const long long grid = (a.n + D::V - 1) / D::V;
    ekf_kernel<MODEL, INTEG><<<(unsigned)grid, D::THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_ekf(int model, int integ, const EkfArgs& a, cudaStream_t st) {
    switch (model) {
        case MODEL_THRUSTER8:
            return integ == INTEG_RK4 ? ekf_go<MODEL_THRUSTER8, INTEG_RK4>(a, st) : ekf_go<MODEL_THRUSTER8, INTEG_EULER>(a, st);
        case MODEL_WRENCH12:
            return integ == INTEG_RK4 ? ekf_go<MODEL_WRENCH12, INTEG_RK4>(a, st) : ekf_go<MODEL_WRENCH12, INTEG_EULER>(a, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace brov
