// brov_device.cuh — device-side BlueROV2 Fossen dynamics, written for one-thread-per-vehicle execution on sm_100a.
//
// Everything a vehicle needs between two HBM touches lives in registers: the 12/13-state vector, the RK4
// accumulator and stage state, the 8x3 thruster-lag state (or the 6 filtered wrench components).  Constants
// reach the FP pipes as constant-bank operands (they are members of the __grid_constant__ kernel argument), or,
// for Monte-Carlo ensembles, from a per-block shared-memory table laid out [param][thread] (conflict-free).
//
// Reference behaviour restated here (file:line in ViktorNfa/bluerov2_dynamics):
//   rotation / Euler-rate kinematics        fossen/BlueROV2.py:23-62
//   T200 polynomial                         fossen/BlueROV2.py:251-257
//   ThrusterLag.step (x <- Ad x + Bd u)     fossen/BlueROV2.py:503-510   (advanced once per dynamics() call)
//   allocation  tau = sum F_i [e_i; r_i x e_i]   fossen/BlueROV2.py:265-278
//   C(nu) nu, D(nu_r) nu_r, g(eta)          fossen/BlueROV2.py:280-355
//   nu_dot = Minv (tau - C nu - D nu_r - g) fossen/BlueROV2.py:390-391
//   quaternion kinematics                   fossen/BlueROV2_wrench.py:27-80,322-367
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

// Layout alternatives measured and rejected in round 1 (lag state / RK4 accumulator in shared memory, 64-thread fp64
// blocks, re-based constant loads, a rolled stage loop, packed FFMA2 fp32 step) are recorded with their timings in
// profiles/r01e_fp64_const_variants.json, r01g_tune_variants.json and DESIGN.md; their code left the tree in round 2.

namespace brov {

// ---------------------------------------------------------------------------------------------------------------
// kernel-parameter vector (derived coefficients; see brov_derive_params in brov_api.cu and include/brov.h)
// ---------------------------------------------------------------------------------------------------------------
enum : int {
    KP_MINV = 0,   // 6: 1/(m - X_udot) ... 1/(Iz - N_rdot)
    KP_A = 6,      // 3: a1 = m - X_udot, a2 = m - Y_vdot, a3 = m - Z_wdot
    KP_DA = 9,     // 3: a3-a2, a1-a3, a2-a1
    KP_DB = 12,    // 3: b3-b2, b1-b3, b2-b1   (b = I - K_pdot ...)
    KP_DL = 15,    // 6: -X_u ...   (linear damping, positive)
    KP_DQ = 21,    // 6: -X_|u|u ... (quadratic damping, positive)
    KP_WMB = 27,   // W - B
    KP_XBB = 28,   // xb*B, yb*B, zb*B
    KP_CUR = 31,   // 3: current velocity, NED
    KP_ILAG1 = 34, // 1 / T_lag of the optional first-order wrench lag (extension)
    KP_COUNT = 36
};

constexpr int MODEL_THRUSTER8 = 0;
constexpr int MODEL_WRENCH12 = 1;
constexpr int MODEL_QUAT13 = 2;
// Double-integrator comparison model (training/train_tank_brov2_rk4.py:461-528 and the Euler twins): kinematics as the
// Fossen models (position through R(eta); Euler angles integrated from the body rates DIRECTLY, no J2), accelerations
// a learned linear map of the input, [v_dot, w_dot] = u [K_lin | K_ang].
constexpr int MODEL_DI12_U8 = 3;    // 12-state, 8 thruster inputs
constexpr int MODEL_DI12_U6 = 4;    // 12-state, 6 wrench inputs
constexpr int MODEL_DIQ13_U6 = 5;   // 13-state quaternion, 6 wrench inputs
constexpr int INTEG_RK4 = 0;
constexpr int INTEG_EULER = 1;

template <int MODEL> struct ModelDim {
    static constexpr bool QUAT = (MODEL == MODEL_QUAT13) || (MODEL == MODEL_DIQ13_U6);
    static constexpr bool DI = (MODEL == MODEL_DI12_U8) || (MODEL == MODEL_DI12_U6) || (MODEL == MODEL_DIQ13_U6);
    static constexpr int NX = QUAT ? 13 : 12;
    static constexpr int NU = (MODEL == MODEL_THRUSTER8 || MODEL == MODEL_DI12_U8) ? 8 : 6;
    static constexpr int NLAG = (MODEL == MODEL_THRUSTER8) ? 24 : 6;  // hidden state per vehicle
    static constexpr int VOFF = QUAT ? 7 : 6;                          // offset of nu in the state
};

// Constants shared by every vehicle of a launch.  Lives in the kernel argument => constant bank 0.
template <typename T> struct Consts {
    T kp[KP_COUNT];
    T alloc[6][8];   // tau = alloc * F; double-integrator engines: alloc[r][i] = [K_lin | K_ang][i][r] (dense)
    // closed-form 3rd-order lag over the NSUB dynamics() calls of one integrator step with the input held:
    //   y_j = lagG[j] . x + lagH[j] * F   (output seen by sub-step j, j = 0..NSUB-1)
    //   x  <- lagA x + lagB F             (state after all NSUB sub-steps)
    T lagG[4][3];
    T lagH[4];
    T lagA[3][3];
    T lagB[3];
    T dt;
    // literal tables of the fp64 build (filled by make_consts): T200 polynomial, sincos kernel, stage-rotation Taylor
    // coefficients.  As kernel-argument members they are fetched with one LDCU.64 each; as C++ literals every use costs
    // two UMOVs, as a __constant__ array they are hoisted into registers and shuffled back through R2UR.
    T poly[5];     // -140.3, 389.9, -404.1, 176.0, 8.9
    T sc[16];      // see kSinCos64
    T rot[8];      // sin: -1/6, 1/120, -1/5040 ; cos: -1/2, 1/24, -1/720, 1/40320 ; pad
    int has_current;
    int use_lag1;
};

// ---------------------------------------------------------------------------------------------------------------
// scalar helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float abs_(float a) { return fabsf(a); }
__device__ __forceinline__ double abs_(double a) { return fabs(a); }
__device__ __forceinline__ float sqrt_(float a) { return sqrtf(a); }
__device__ __forceinline__ double sqrt_(double a) { return sqrt(a); }

// 1/a.  fp32: MUFU.RCP seed + one Newton step (<= 1 ulp for normal a); inf/0 behave like IEEE division.
__device__ __forceinline__ float rcp_(float a) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    float e = fmaf(-a, r, 1.0f);
    float r2 = fmaf(r, e, r);
    // keep the seed when the Newton step degenerates (a = 0 or inf: e is NaN)
    return (e == e) ? r2 : r;
}
// fp64: MUFU.RCP64H seed (2^-23 relative) + two Newton steps with an FMA residual (<= 1 ulp for normal a); zeros,
// infinities, NaNs and denormal-range operands take the IEEE division.
__device__ __forceinline__ double rcp_(double a) {
    const double aa = fabs(a);
    if (!(aa > 1e-290 && aa < 1e290)) return 1.0 / a;
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    r = fma(r, fma(-a, r, 1.0), r);
    r = fma(r, fma(-a, r, 1.0), r);
    return r;
}

// 1/a without the range guard, for operands known to be normal and far from the ends of the exponent range (clamped
// cosines >= 1e-7, quaternion norms >= 1e-12): no branch in the step
__device__ __forceinline__ float rcp_nr(float a) { return rcp_(a); }
__device__ __forceinline__ double rcp_nr(double a) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    r = fma(r, fma(-a, r, 1.0), r);
    r = fma(r, fma(-a, r, 1.0), r);
    return r;
}

// sin & cos.  fp32: 3-term Cody-Waite reduction by pi/2 (FMA keeps the products exact) + minimax polynomials on
// [-pi/4, pi/4] (Cephes sinf/cosf coefficients); |error| <= ~1.5 ulp.  No slow path, no local memory; domain
// |a| < 2^30 rad (a float that large has an ulp of 64 rad anyway).
__device__ __forceinline__ void sincos_(float a, float* s, float* c, const float* = nullptr) {
    float j = rintf(a * 0.6366197466850281f);
    float r = fmaf(-j, 1.5707963705062866f, a);
    r = fmaf(-j, -4.371138828673793e-08f, r);
    r = fmaf(-j, -1.7151245100058819e-15f, r);
    int q = (int)j;
    float z = r * r;
    float ps = fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f);
    float sn = fmaf(ps * z, r, r);
    float pc = fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f);
    float cs = fmaf(pc * z, z, fmaf(-0.5f, z, 1.0f));
    float ss = (q & 1) ? cs : sn;
    float cc = (q & 1) ? sn : cs;
    *s = (q & 2) ? -ss : ss;
    *c = ((q + 1) & 2) ? -cc : cc;
}
// [0] 2/pi, [1..3] pi/2 in three parts, [4..9] sin coefficients S1..S6, [10..15] cos coefficients C1..C6 (fdlibm)
static __constant__ double kSinCos64[16] = {
    0.6366197723675814, 1.5707963267948966, 6.123233995736766e-17, -1.4973849048591698e-33,
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04,
    2.75573137070700676789e-06, -2.50507602534068634195e-08, 1.58969099521155010221e-10,
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05,
    -2.75573143513906633035e-07, 2.08757232129817482790e-09, -1.13596475577881948265e-11};
// fp64: same scheme with the fdlibm __kernel_sin/__kernel_cos coefficients.  The FMA makes each reduction step a
// single rounding, so full-precision parts of pi/2 suffice.  Domain |a| < 2^30 rad (quadrant held in an int).
__device__ __forceinline__ void sincos_(double a, double* s, double* c, const double* K = kSinCos64) {
    double j = rint(a * K[0]);
    double r = fma(-j, K[1], a);
    r = fma(-j, K[2], r);
    r = fma(-j, K[3], r);
    int q = (int)j;
    double z = r * r;
    double ps = fma(fma(fma(fma(K[9], z, K[8]), z, K[7]), z, K[6]), z, K[5]);
    ps = fma(ps, z, K[4]);
    double sn = fma(ps * z, r, r);
    double pc = fma(fma(fma(fma(K[15], z, K[14]), z, K[13]), z, K[12]), z, K[11]);
    pc = fma(pc, z, K[10]);
    double cs = fma(pc * z, z, fma(-0.5, z, 1.0));
    double ss = (q & 1) ? cs : sn;
    double cc = (q & 1) ? sn : cs;
    *s = (q & 2) ? -ss : ss;
    *c = ((q + 1) & 2) ? -cc : cc;
}

// ---------------------------------------------------------------------------------------------------------------
// parameter access: constant bank (shared by all vehicles) or shared-memory table (per-vehicle Monte-Carlo)
// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct ParamsConst {
    const T* kp;  // points into the __grid_constant__ argument
    __device__ __forceinline__ T operator[](int i) const { return kp[i]; }
};
template <typename T> struct ParamsShared {
    const T* base;  // &table[0][threadIdx.x]
    int pitch;      // blockDim.x
    __device__ __forceinline__ T operator[](int i) const { return base[i * pitch]; }
};
// per-vehicle coefficients held in registers for the whole launch (fp32 Monte-Carlo rollouts: every coefficient is used
// once per RHS evaluation, i.e. the shared-memory table costs ~130 LDS per RK4 step; indices are compile-time constants
// after unrolling, unused entries are dropped by the compiler)
template <typename T> struct ParamsRegs {
    T v[KP_COUNT];
    __device__ __forceinline__ T operator[](int i) const { return v[i]; }
};

// ---------------------------------------------------------------------------------------------------------------
// model pieces
// ---------------------------------------------------------------------------------------------------------------

// T200 static thrust curve, Horner in V^2 (fossen/BlueROV2.py:251-257; the reference uses pow(), <= 3 ulp apart).
template <typename T> __device__ __forceinline__ T thrust_poly(T V) {
    T z = V * V;
    T p = T(-140.3) * z + T(389.9);
    p = p * z + T(-404.1);
    p = p * z + T(176.0);
    p = p * z + T(8.9);
    return p * V;
}
// same with the coefficients read from the constant block (fp64 rollouts)
template <typename T> __device__ __forceinline__ T thrust_poly(const Consts<T>& c, T V) {
    if constexpr (sizeof(T) == 8) {
        T z = V * V;
        T p = c.poly[0] * z + c.poly[1];
        p = p * z + c.poly[2];
        p = p * z + c.poly[3];
        p = p * z + c.poly[4];
        return p * V;
    } else {
        return thrust_poly<T>(V);
    }
}

// dF/dV of the T200 curve F(V) = V p(V^2): 9 a z^4 + 7 b z^3 + 5 c z^2 + 3 d z + e with z = V^2
__device__ __forceinline__ double thrust_poly_d(const Consts<double>& c, double V) {
    const double z = V * V;
    double p = 9.0 * c.poly[0] * z + 7.0 * c.poly[1];
    p = p * z + 5.0 * c.poly[2];
    p = p * z + 3.0 * c.poly[3];
    return p * z + c.poly[4];
}

// nu_dot = Minv (tau - C(nu) nu - D(nu_r) nu_r - g); g from (sin th, cos th sin phi, cos th cos phi).
// Every axis is ONE chain of fused multiply-adds onto tau_i: the Coriolis terms (closed form of C_RB + C_A times nu,
// fossen/BlueROV2.py:280-325), the restoring terms (:340-355) and the damping term (:327-338) are accumulated with
// their signs instead of being formed as separate vectors and subtracted (47 instead of 62 operations; measured
// against the separate-vector form, profiles/r02h_tune_variants.txt: fp32 thruster rollout 3.02 against 3.07 ms,
// fp64 4.51 against 4.48 ms per 1000 steps — kept for both).
template <typename T, class P>
__device__ __forceinline__ void nu_dot(const T* __restrict__ nu, const T* __restrict__ nur, const T* __restrict__ tau,
                                       T sth, T cs, T cc, const P& p, T* __restrict__ out) {
    const T u = nu[0], v = nu[1], w = nu[2], pp = nu[3], q = nu[4], r = nu[5];
    const T a1u = p[KP_A + 0] * u, a2v = p[KP_A + 1] * v, a3w = p[KP_A + 2] * w;
    const T wmb = p[KP_WMB], xbB = p[KP_XBB + 0], ybB = p[KP_XBB + 1], zbB = p[KP_XBB + 2];
    T t[6];
    // [C nu]_0 = a3 w q - a2 v r          g_0 = (W-B) sin th
    t[0] = tau[0] - a3w * q;   t[0] += a2v * r;   t[0] -= wmb * sth;
    // [C nu]_1 = a1 u r - a3 w p          g_1 = -(W-B) cos th sin phi
    t[1] = tau[1] - a1u * r;   t[1] += a3w * pp;  t[1] += wmb * cs;
    // [C nu]_2 = a2 v p - a1 u q          g_2 = -(W-B) cos th cos phi
    t[2] = tau[2] - a2v * pp;  t[2] += a1u * q;   t[2] += wmb * cc;
    // [C nu]_3 = (a3-a2) v w + (b3-b2) q r     g_3 = yb B cc - zb B cs
    t[3] = tau[3] - p[KP_DA + 0] * (v * w);  t[3] -= p[KP_DB + 0] * (q * r);   t[3] -= ybB * cc;  t[3] += zbB * cs;
    // [C nu]_4 = (a1-a3) u w + (b1-b3) p r     g_4 = -zb B sth - xb B cc
    t[4] = tau[4] - p[KP_DA + 1] * (u * w);  t[4] -= p[KP_DB + 1] * (pp * r);  t[4] += zbB * sth; t[4] += xbB * cc;
    // [C nu]_5 = (a2-a1) u v + (b2-b1) p q     g_5 = xb B cs + yb B sth
    t[5] = tau[5] - p[KP_DA + 2] * (u * v);  t[5] -= p[KP_DB + 2] * (pp * q);  t[5] -= xbB * cs;  t[5] -= ybB * sth;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        T d = p[KP_DQ + i] * abs_(nur[i]) + p[KP_DL + i];
        out[i] = p[KP_MINV + i] * (t[i] - d * nur[i]);
    }
}

// Reverse mode of nu_dot (fp64): g[6] is the cotangent of out.  Returns the cotangents of nu (gnu), of nur (gnur), of
// the three restoring-term inputs (sth, cs, cc) and of tau (gtau).  Branch taken: d|x| = sign(x) dx, sign(0) = 0.
template <class P>
__device__ __forceinline__ void nu_dot_vjp(const double* __restrict__ nu, const double* __restrict__ nur, const P& p,
                                           const double* __restrict__ g, double* __restrict__ gnu,
                                           double* __restrict__ gnur, double& gsth, double& gcs, double& gcc,
                                           double* __restrict__ gtau) {
    const double u = nu[0], v = nu[1], w = nu[2], pp = nu[3], q = nu[4], r = nu[5];
    const double a1u = p[KP_A + 0] * u, a2v = p[KP_A + 1] * v, a3w = p[KP_A + 2] * w;
    const double wmb = p[KP_WMB], xbB = p[KP_XBB + 0], ybB = p[KP_XBB + 1], zbB = p[KP_XBB + 2];
    double e[6];   // cotangent of t[i] (= of tau[i])
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        e[i] = p[KP_MINV + i] * g[i];
        gtau[i] = e[i];
        // d(d_i nur_i) / d nur_i = 2 DQ_i |nur_i| + DL_i
        const double s = nur[i] > 0.0 ? 1.0 : (nur[i] < 0.0 ? -1.0 : 0.0);
        const double dd = p[KP_DQ + i] * abs_(nur[i]) + p[KP_DL + i] + p[KP_DQ + i] * s * nur[i];
        gnur[i] = -e[i] * dd;
    }
    const double ga1u = q * e[2] - r * e[1], ga2v = r * e[0] - pp * e[2], ga3w = pp * e[1] - q * e[0];
    gnu[0] = p[KP_A + 0] * ga1u - p[KP_DA + 1] * w * e[4] - p[KP_DA + 2] * v * e[5];
    gnu[1] = p[KP_A + 1] * ga2v - p[KP_DA + 0] * w * e[3] - p[KP_DA + 2] * u * e[5];
    gnu[2] = p[KP_A + 2] * ga3w - p[KP_DA + 0] * v * e[3] - p[KP_DA + 1] * u * e[4];
    gnu[3] = a3w * e[1] - a2v * e[2] - p[KP_DB + 1] * r * e[4] - p[KP_DB + 2] * q * e[5];
    gnu[4] = a1u * e[2] - a3w * e[0] - p[KP_DB + 0] * r * e[3] - p[KP_DB + 2] * pp * e[5];
    gnu[5] = a2v * e[0] - a1u * e[1] - p[KP_DB + 0] * q * e[3] - p[KP_DB + 1] * pp * e[4];
    gsth = zbB * e[4] - wmb * e[0] - ybB * e[5];
    gcs = wmb * e[1] + zbB * e[3] - xbB * e[5];
    gcc = wmb * e[2] - ybB * e[3] + xbB * e[4];
}

// Coefficient cotangent of nu_dot (fp64) at (nu, nur, tau, sth, cs, cc) with the cotangent g[6] of out: adds
// d<g, out>/d kp to gk[KP_MINV .. KP_XBB + 2] (the current enters through nur: rhs_euler12_vjp / rhs_quat13_vjp add
// gk[KP_CUR ..]).  gk is any indexable accumulator of doubles (a shared-memory column in the adjoint kernel).
template <class P, class G>
__device__ __forceinline__ void nu_dot_coef_vjp(const double* __restrict__ nu, const double* __restrict__ nur,
                                                const double* __restrict__ tau, double sth, double cs, double cc,
                                                const P& p, const double* __restrict__ g, const G& gk) {
    const double u = nu[0], v = nu[1], w = nu[2], pp = nu[3], q = nu[4], r = nu[5];
    const double a1u = p[KP_A + 0] * u, a2v = p[KP_A + 1] * v, a3w = p[KP_A + 2] * w;
    const double wmb = p[KP_WMB], xbB = p[KP_XBB + 0], ybB = p[KP_XBB + 1], zbB = p[KP_XBB + 2];
    double t[6], e[6];
    t[0] = tau[0] - a3w * q + a2v * r - wmb * sth;
    t[1] = tau[1] - a1u * r + a3w * pp + wmb * cs;
    t[2] = tau[2] - a2v * pp + a1u * q + wmb * cc;
    t[3] = tau[3] - p[KP_DA + 0] * (v * w) - p[KP_DB + 0] * (q * r) - ybB * cc + zbB * cs;
    t[4] = tau[4] - p[KP_DA + 1] * (u * w) - p[KP_DB + 1] * (pp * r) + zbB * sth + xbB * cc;
    t[5] = tau[5] - p[KP_DA + 2] * (u * v) - p[KP_DB + 2] * (pp * q) - xbB * cs - ybB * sth;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        e[i] = p[KP_MINV + i] * g[i];
        const double an = abs_(nur[i]);
        gk[KP_MINV + i] += g[i] * (t[i] - (p[KP_DQ + i] * an + p[KP_DL + i]) * nur[i]);
        gk[KP_DL + i] -= e[i] * nur[i];
        gk[KP_DQ + i] -= e[i] * an * nur[i];
    }
    gk[KP_A + 0] += u * (q * e[2] - r * e[1]);
    gk[KP_A + 1] += v * (r * e[0] - pp * e[2]);
    gk[KP_A + 2] += w * (pp * e[1] - q * e[0]);
    gk[KP_DA + 0] -= v * w * e[3];
    gk[KP_DA + 1] -= u * w * e[4];
    gk[KP_DA + 2] -= u * v * e[5];
    gk[KP_DB + 0] -= q * r * e[3];
    gk[KP_DB + 1] -= pp * r * e[4];
    gk[KP_DB + 2] -= pp * q * e[5];
    gk[KP_WMB] += cs * e[1] + cc * e[2] - sth * e[0];
    gk[KP_XBB + 0] += cc * e[4] - cs * e[5];
    gk[KP_XBB + 1] -= cc * e[3] + sth * e[5];
    gk[KP_XBB + 2] += cs * e[3] + sth * e[4];
}

// Euler-angle models: xdot[12] from x[12] and the body wrench tau[6].
template <typename T> struct Trig { T sphi, cphi, sth, cth, spsi, cpsi; };

template <typename T> __device__ __forceinline__ void trig_full(const T* __restrict__ ang, Trig<T>& t) {
    sincos_(ang[0], &t.sphi, &t.cphi);
    sincos_(ang[1], &t.sth, &t.cth);
    sincos_(ang[2], &t.spsi, &t.cpsi);
}
template <typename T>
__device__ __forceinline__ void trig_full(const Consts<T>& c, const T* __restrict__ ang, Trig<T>& t) {
    if constexpr (sizeof(T) == 8) {
        sincos_(ang[0], &t.sphi, &t.cphi, c.sc);
        sincos_(ang[1], &t.sth, &t.cth, c.sc);
        sincos_(ang[2], &t.spsi, &t.cpsi, c.sc);
    } else {
        trig_full<T>(ang, t);
    }
}

// fp32 RK4 stages 2..4: the stage angles are base + d with a small increment d = c*dt*k, so their sines/cosines
// follow from the step's base values by the angle-addition formulas with a short Taylor series for sin d, cos d
// (|d| <= 1/8: truncation < 1e-9 relative, i.e. below float rounding): 11 instructions per angle instead of ~26 for
// a full range-reduced sincos.  Larger increments (angular rate > 6 rad/s at dt = 0.02) take the full path.
// It evaluates sin/cos of the UNROUNDED sum base + d, which is closer to exact arithmetic than sin(fl(base + d)).
__device__ __forceinline__ void rotate_sc(float s, float c, float d, float* so, float* co) {
    float z = d * d;
    float sd = fmaf(d * z, fmaf(z, 8.3333333e-3f, -1.6666667e-1f), d);
    float cd = fmaf(z, fmaf(z, fmaf(z, -1.3888889e-3f, 4.1666667e-2f), -0.5f), 1.0f);
    *so = fmaf(s, cd, c * sd);
    *co = fmaf(c, cd, -(s * sd));
}
__device__ __forceinline__ void trig_stage(const Consts<float>&, const Trig<float>& b, const float* __restrict__ d,
                                           const float* __restrict__ ang, Trig<float>& t) {
    if (fmaxf(fmaxf(fabsf(d[0]), fabsf(d[1])), fabsf(d[2])) > 0.125f) {
        trig_full<float>(ang, t);
    } else {
        rotate_sc(b.sphi, b.cphi, d[0], &t.sphi, &t.cphi);
        rotate_sc(b.sth, b.cth, d[1], &t.sth, &t.cth);
        rotate_sc(b.spsi, b.cpsi, d[2], &t.spsi, &t.cpsi);
    }
}
// fp64: same idea with two more Taylor terms and a tighter bound (|d| <= 1/32: truncation < 1e-19 relative); the
// result differs from a full evaluation by ~2 ulp, 6 orders of magnitude inside the 1e-10 parity budget.
__device__ __forceinline__ void rotate_sc(const double* __restrict__ K, double s, double c, double d, double* so,
                                          double* co) {
    double z = d * d;
    double sd = fma(d * z, fma(z, fma(z, K[2], K[1]), K[0]), d);
    double cd = fma(z, fma(z, fma(z, fma(z, K[6], K[5]), K[4]), K[3]), 1.0);
    *so = fma(s, cd, c * sd);
    *co = fma(c, cd, -(s * sd));
}
__device__ __forceinline__ void trig_stage(const Consts<double>& c, const Trig<double>& b, const double* __restrict__ d,
                                           const double* __restrict__ ang, Trig<double>& t) {
    // |d| > 1/32 decided on the high words (integer pipe: the FP64 pipe is the one this kernel is short of)
    const int h0 = __double2hiint(d[0]) & 0x7fffffff, h1 = __double2hiint(d[1]) & 0x7fffffff, h2 = __double2hiint(d[2]) & 0x7fffffff;
    if (max(max(h0, h1), h2) > 0x3FA00000) {
        trig_full<double>(c, ang, t);
    } else {
        rotate_sc(c.rot, b.sphi, b.cphi, d[0], &t.sphi, &t.cphi);
        rotate_sc(c.rot, b.sth, b.cth, d[1], &t.sth, &t.cth);
        rotate_sc(c.rot, b.spsi, b.cpsi, d[2], &t.spsi, &t.cpsi);
    }
}

template <typename T, class P>
__device__ __forceinline__ void rhs_euler12(const T* __restrict__ x, const Trig<T>& tr, const T* __restrict__ tau,
                                            const P& p, bool has_current, T* __restrict__ xd) {
    const T sphi = tr.sphi, cphi = tr.cphi, sth = tr.sth, cth = tr.cth, spsi = tr.spsi, cpsi = tr.cpsi;
    const T* nu = x + 6;
    // p_dot = Rz(psi) Ry(theta) Rx(phi) nu_1 as three planar rotations
    {
        T v1 = cphi * nu[1] - sphi * nu[2];
        T w1 = sphi * nu[1] + cphi * nu[2];
        T u2 = cth * nu[0] + sth * w1;
        xd[2] = cth * w1 - sth * nu[0];
        xd[0] = cpsi * u2 - spsi * v1;
        xd[1] = spsi * u2 + cpsi * v1;
    }
    // Euler rates with the reference's cos(theta) clamp: |c| < 1e-7 -> 1e-7 * sign(c), sign(0) = 0
    {
        T ct = cth;
        // The clamp and the division by zero are decided exactly, but only inside a rarely taken branch entered on a
        // cheap test (fp64: an integer compare of the high word against that of 1e-7): four FP compares and their
        // selects per stage otherwise sit on the critical pipe (measured r02t: fp64 +1.4 %, fp32 +3.3 %).
        T ic;
        bool near0;
        if constexpr (sizeof(T) == 8) near0 = (__double2hiint(ct) & 0x7fffffff) <= 0x3E7AD7F2;   // high word of 1e-7
        else near0 = abs_(ct) < T(1e-7);
        if (near0) {
            if (abs_(ct) < T(1e-7)) ct = (ct > T(0)) ? T(1e-7) : ((ct < T(0)) ? T(-1e-7) : T(0));
            // |ct| >= 1e-7, or exactly +0 (sign(0) = 0), where the reference divides by zero: 1 / +0 = +inf
            ic = (ct == T(0)) ? T(INFINITY) : rcp_nr(ct);
        } else {
            ic = rcp_nr(ct);
        }
        T sq = sphi * nu[4] + cphi * nu[5];
        T psd = sq * ic;
        xd[5] = psd;
        xd[4] = cphi * nu[4] - sphi * nu[5];
        xd[3] = nu[3] + sth * psd;
    }
    T nur[6] = {nu[0], nu[1], nu[2], nu[3], nu[4], nu[5]};
    if (has_current) {  // nu_r = nu - R^T v_c  (inverse rotations in the opposite order)
        T cx = p[KP_CUR + 0], cy = p[KP_CUR + 1], cz = p[KP_CUR + 2];
        T x1 = cpsi * cx + spsi * cy;
        T y1 = cpsi * cy - spsi * cx;
        T x2 = cth * x1 - sth * cz;
        T z2 = sth * x1 + cth * cz;
        T y3 = cphi * y1 + sphi * z2;
        T z3 = cphi * z2 - sphi * y1;
        nur[0] -= x2;
        nur[1] -= y3;
        nur[2] -= z3;
    }
    nu_dot<T>(nu, nur, tau, sth, cth * sphi, cth * cphi, p, xd + 6);
}

// Reverse mode of rhs_euler12 (fp64) at (x, tau) with the sines and cosines tr of x[3..5]: g[12] is the cotangent of
// xd; a[12] receives the cotangent of x and gtau[6] that of tau.  Same convention as the dual instantiation of
// rhs_euler12: the clamped cos(theta) (|c| < 1e-7) is a constant, otherwise d(1/c) = -dc / c^2.
// COEF: also adds the coefficient cotangent to gk (nu_dot_coef_vjp at the wrench tau, and gk[KP_CUR ..] = -R gnur,
// which needs has_current: with a zero current nu - R^T 0 = nu, so the primal is unchanged).
template <bool COEF = false, class P, class G = double*>
__device__ __forceinline__ void rhs_euler12_vjp(const double* __restrict__ x, const Trig<double>& tr,
                                                const P& p, bool has_current, const double* __restrict__ g,
                                                double* __restrict__ a, double* __restrict__ gtau,
                                                const double* __restrict__ tau = nullptr, const G& gk = G()) {
    const double sphi = tr.sphi, cphi = tr.cphi, sth = tr.sth, cth = tr.cth, spsi = tr.spsi, cpsi = tr.cpsi;
    const double* nu = x + 6;
    double nur[6] = {nu[0], nu[1], nu[2], nu[3], nu[4], nu[5]};
    double cx = 0.0, cy = 0.0, cz = 0.0, x1 = 0.0, y1 = 0.0, z2 = 0.0;
    if (has_current) {
        cx = p[KP_CUR + 0]; cy = p[KP_CUR + 1]; cz = p[KP_CUR + 2];
        x1 = cpsi * cx + spsi * cy;
        y1 = cpsi * cy - spsi * cx;
        const double x2 = cth * x1 - sth * cz;
        z2 = sth * x1 + cth * cz;
        const double y3 = cphi * y1 + sphi * z2;
        const double z3 = cphi * z2 - sphi * y1;
        nur[0] -= x2;
        nur[1] -= y3;
        nur[2] -= z3;
    }
    double gnu[6], gnur[6], gsth, gcs, gcc;
    nu_dot_vjp(nu, nur, p, g + 6, gnu, gnur, gsth, gcs, gcc, gtau);
    if constexpr (COEF) nu_dot_coef_vjp(nu, nur, tau, sth, cth * sphi, cth * cphi, p, g + 6, gk);
    double gsphi = cth * gcs, gcphi = cth * gcc, gcth = sphi * gcs + cphi * gcc, gspsi = 0.0, gcpsi = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) gnu[i] += gnur[i];
    if (has_current) {   // nur[0..2] -= (x2, y3, z3)
        const double gx2 = -gnur[0], gy3 = -gnur[1], gz3 = -gnur[2];
        const double gy1 = cphi * gy3 - sphi * gz3;
        const double gz2 = sphi * gy3 + cphi * gz3;
        gcphi += y1 * gy3 + z2 * gz3;
        gsphi += z2 * gy3 - y1 * gz3;
        const double gx1 = cth * gx2 + sth * gz2;
        gcth += x1 * gx2 + cz * gz2;
        gsth += x1 * gz2 - cz * gx2;
        gcpsi += cx * gx1 + cy * gy1;
        gspsi += cy * gx1 - cx * gy1;
        if constexpr (COEF) {   // x1, y1 = Rz^T c; (x2, z2) = Ry^T (x1, cz)
            gk[KP_CUR + 0] += cpsi * gx1 - spsi * gy1;
            gk[KP_CUR + 1] += spsi * gx1 + cpsi * gy1;
            gk[KP_CUR + 2] += cth * gz2 - sth * gx2;
        }
    }
    // Euler rates
    {
        double ic;
        const bool clamped = fabs(cth) < 1e-7;
        if (clamped) {
            const double ct = (cth > 0.0) ? 1e-7 : ((cth < 0.0) ? -1e-7 : 0.0);
            ic = (ct == 0.0) ? (double)INFINITY : rcp_nr(ct);
        } else {
            ic = rcp_nr(cth);
        }
        const double sq = sphi * nu[4] + cphi * nu[5];
        const double psd = sq * ic;
        gnu[3] += g[3];
        gsth += psd * g[3];
        const double gpsd = g[5] + sth * g[3];
        const double gsq = ic * gpsd;
        if (!clamped) gcth -= ic * ic * (sq * gpsd);
        gsphi += nu[4] * gsq - nu[5] * g[4];
        gcphi += nu[5] * gsq + nu[4] * g[4];
        gnu[4] += sphi * gsq + cphi * g[4];
        gnu[5] += cphi * gsq - sphi * g[4];
    }
    // p_dot = Rz(psi) Ry(theta) Rx(phi) nu_1
    {
        const double v1 = cphi * nu[1] - sphi * nu[2];
        const double w1 = sphi * nu[1] + cphi * nu[2];
        const double u2 = cth * nu[0] + sth * w1;
        const double gu2 = cpsi * g[0] + spsi * g[1];
        const double gv1 = cpsi * g[1] - spsi * g[0];
        gcpsi += u2 * g[0] + v1 * g[1];
        gspsi += u2 * g[1] - v1 * g[0];
        const double gw1 = cth * g[2] + sth * gu2;
        gnu[0] += cth * gu2 - sth * g[2];
        gcth += w1 * g[2] + nu[0] * gu2;
        gsth += w1 * gu2 - nu[0] * g[2];
        gnu[1] += cphi * gv1 + sphi * gw1;
        gnu[2] += cphi * gw1 - sphi * gv1;
        gcphi += nu[1] * gv1 + nu[2] * gw1;
        gsphi += nu[1] * gw1 - nu[2] * gv1;
    }
    a[0] = 0.0; a[1] = 0.0; a[2] = 0.0;
    a[3] = cphi * gsphi - sphi * gcphi;
    a[4] = cth * gsth - sth * gcth;
    a[5] = cpsi * gspsi - spsi * gcpsi;
#pragma unroll
    for (int i = 0; i < 6; ++i) a[6 + i] = gnu[i];
}

// Quaternion model: xdot[13] from x[13] = [pos, qw qx qy qz, nu] (fossen/BlueROV2_wrench.py:322-367).
template <typename T, class P>
__device__ __forceinline__ void rhs_quat13(const T* __restrict__ x, const T* __restrict__ tau, const P& p,
                                           bool has_current, T* __restrict__ xd) {
    T qw = x[3], qx = x[4], qy = x[5], qz = x[6];
    {
        T n2 = qw * qw + qx * qx + qy * qy + qz * qz;
        T n = sqrt_(n2);
        if (n < T(1e-12)) { qw = T(1); qx = qy = qz = T(0); }
        else { T in = rcp_nr(n); qw *= in; qx *= in; qy *= in; qz *= in; }
    }
    const T* nu = x + 7;
    T R00 = T(1) - T(2) * (qy * qy + qz * qz), R01 = T(2) * (qx * qy - qz * qw), R02 = T(2) * (qx * qz + qy * qw);
    T R10 = T(2) * (qx * qy + qz * qw), R11 = T(1) - T(2) * (qx * qx + qz * qz), R12 = T(2) * (qy * qz - qx * qw);
    T R20 = T(2) * (qx * qz - qy * qw), R21 = T(2) * (qy * qz + qx * qw), R22 = T(1) - T(2) * (qx * qx + qy * qy);
    xd[0] = R00 * nu[0] + R01 * nu[1] + R02 * nu[2];
    xd[1] = R10 * nu[0] + R11 * nu[1] + R12 * nu[2];
    xd[2] = R20 * nu[0] + R21 * nu[1] + R22 * nu[2];
    const T wp = nu[3], wq = nu[4], wr = nu[5];
    xd[3] = T(0.5) * (-qx * wp - qy * wq - qz * wr);
    xd[4] = T(0.5) * (qw * wp + qy * wr - qz * wq);
    xd[5] = T(0.5) * (qw * wq - qx * wr + qz * wp);
    xd[6] = T(0.5) * (qw * wr + qx * wq - qy * wp);
    T nur[6] = {nu[0], nu[1], nu[2], nu[3], nu[4], nu[5]};
    if (has_current) {
        T cx = p[KP_CUR + 0], cy = p[KP_CUR + 1], cz = p[KP_CUR + 2];
        nur[0] -= R00 * cx + R10 * cy + R20 * cz;
        nur[1] -= R01 * cx + R11 * cy + R21 * cz;
        nur[2] -= R02 * cx + R12 * cy + R22 * cz;
    }
    nu_dot<T>(nu, nur, tau, -R20, R21, R22, p, xd + 7);
}

// Reverse mode of the normalisation q -> q / |q| at a raw q with |q| >= 1e-12: g[4] (cotangent of the unit
// quaternion) is replaced by that of the raw one, (g - y (y . g)) / |q| with y = q / |q|.  Below 1e-12 the fallback
// (1, 0, 0, 0) is a constant: the cotangent is zero.
__device__ __forceinline__ void quat_normalize_vjp(const double* __restrict__ q, double* __restrict__ g) {
    const double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n < 1e-12) { g[0] = g[1] = g[2] = g[3] = 0.0; return; }
    const double in = rcp_nr(n);
    const double y0 = q[0] * in, y1 = q[1] * in, y2 = q[2] * in, y3 = q[3] * in;
    const double yg = y0 * g[0] + y1 * g[1] + y2 * g[2] + y3 * g[3];
    g[0] = (g[0] - y0 * yg) * in;
    g[1] = (g[1] - y1 * yg) * in;
    g[2] = (g[2] - y2 * yg) * in;
    g[3] = (g[3] - y3 * yg) * in;
}

// Reverse mode of rhs_quat13 (fp64) at (x, tau): g[13] is the cotangent of xd; a[13] receives the cotangent of x and
// gtau[6] that of tau.  The quaternion is normalised inside the right-hand side, so its cotangent passes through
// quat_normalize_vjp.  COEF: as rhs_euler12_vjp.
template <bool COEF = false, class P, class G = double*>
__device__ __forceinline__ void rhs_quat13_vjp(const double* __restrict__ x, const P& p, bool has_current,
                                               const double* __restrict__ g, double* __restrict__ a,
                                               double* __restrict__ gtau, const double* __restrict__ tau = nullptr,
                                               const G& gk = G()) {
    double qw = x[3], qx = x[4], qy = x[5], qz = x[6];
    {
        const double n = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
        if (n < 1e-12) { qw = 1.0; qx = qy = qz = 0.0; }
        else { const double in = rcp_nr(n); qw *= in; qx *= in; qy *= in; qz *= in; }
    }
    const double* nu = x + 7;
    const double R00 = 1.0 - 2.0 * (qy * qy + qz * qz), R01 = 2.0 * (qx * qy - qz * qw), R02 = 2.0 * (qx * qz + qy * qw);
    const double R10 = 2.0 * (qx * qy + qz * qw), R11 = 1.0 - 2.0 * (qx * qx + qz * qz), R12 = 2.0 * (qy * qz - qx * qw);
    const double R20 = 2.0 * (qx * qz - qy * qw), R21 = 2.0 * (qy * qz + qx * qw), R22 = 1.0 - 2.0 * (qx * qx + qy * qy);
    double nur[6] = {nu[0], nu[1], nu[2], nu[3], nu[4], nu[5]};
    double cx = 0.0, cy = 0.0, cz = 0.0;
    if (has_current) {
        cx = p[KP_CUR + 0]; cy = p[KP_CUR + 1]; cz = p[KP_CUR + 2];
        nur[0] -= R00 * cx + R10 * cy + R20 * cz;
        nur[1] -= R01 * cx + R11 * cy + R21 * cz;
        nur[2] -= R02 * cx + R12 * cy + R22 * cz;
    }
    double gnu[6], gnur[6], gsth, gcs, gcc;
    nu_dot_vjp(nu, nur, p, g + 7, gnu, gnur, gsth, gcs, gcc, gtau);
    if constexpr (COEF) nu_dot_coef_vjp(nu, nur, tau, -R20, R21, R22, p, g + 7, gk);
    // restoring terms: sth = -R20, cs = R21, cc = R22
    double gR00 = 0.0, gR01 = 0.0, gR02 = 0.0, gR10 = 0.0, gR11 = 0.0, gR12 = 0.0;
    double gR20 = -gsth, gR21 = gcs, gR22 = gcc;
#pragma unroll
    for (int i = 0; i < 6; ++i) gnu[i] += gnur[i];
    if (has_current) {
        gR00 -= cx * gnur[0]; gR10 -= cy * gnur[0]; gR20 -= cz * gnur[0];
        gR01 -= cx * gnur[1]; gR11 -= cy * gnur[1]; gR21 -= cz * gnur[1];
        gR02 -= cx * gnur[2]; gR12 -= cy * gnur[2]; gR22 -= cz * gnur[2];
        if constexpr (COEF) {   // nur[0..2] -= R^T c
            gk[KP_CUR + 0] -= R00 * gnur[0] + R01 * gnur[1] + R02 * gnur[2];
            gk[KP_CUR + 1] -= R10 * gnur[0] + R11 * gnur[1] + R12 * gnur[2];
            gk[KP_CUR + 2] -= R20 * gnur[0] + R21 * gnur[1] + R22 * gnur[2];
        }
    }
    // position rates xd[0..2] = R nu[0..2]
    gR00 += g[0] * nu[0]; gR01 += g[0] * nu[1]; gR02 += g[0] * nu[2];
    gR10 += g[1] * nu[0]; gR11 += g[1] * nu[1]; gR12 += g[1] * nu[2];
    gR20 += g[2] * nu[0]; gR21 += g[2] * nu[1]; gR22 += g[2] * nu[2];
    gnu[0] += R00 * g[0] + R10 * g[1] + R20 * g[2];
    gnu[1] += R01 * g[0] + R11 * g[1] + R21 * g[2];
    gnu[2] += R02 * g[0] + R12 * g[1] + R22 * g[2];
    // quaternion rates xd[3..6] = 1/2 q (x) [0, w]
    const double wp = nu[3], wq = nu[4], wr = nu[5];
    const double h3 = 0.5 * g[3], h4 = 0.5 * g[4], h5 = 0.5 * g[5], h6 = 0.5 * g[6];
    double gq[4];
    gq[0] = h4 * wp + h5 * wq + h6 * wr;
    gq[1] = h6 * wq - h3 * wp - h5 * wr;
    gq[2] = h4 * wr - h3 * wq - h6 * wp;
    gq[3] = h5 * wp - h3 * wr - h4 * wq;
    gnu[3] += qw * h4 + qz * h5 - qx * h3 - qy * h6;
    gnu[4] += qw * h5 + qx * h6 - qy * h3 - qz * h4;
    gnu[5] += qw * h6 + qy * h4 - qz * h3 - qx * h5;
    // rotation matrix entries -> unit quaternion
    gq[0] += 2.0 * (qz * (gR10 - gR01) + qy * (gR02 - gR20) + qx * (gR21 - gR12));
    gq[1] += 2.0 * (qy * (gR01 + gR10) + qz * (gR02 + gR20) + qw * (gR21 - gR12)) - 4.0 * qx * (gR11 + gR22);
    gq[2] += 2.0 * (qx * (gR01 + gR10) + qw * (gR02 - gR20) + qz * (gR12 + gR21)) - 4.0 * qy * (gR00 + gR22);
    gq[3] += 2.0 * (qw * (gR10 - gR01) + qx * (gR02 + gR20) + qy * (gR12 + gR21)) - 4.0 * qz * (gR00 + gR11);
    quat_normalize_vjp(x + 3, gq);
    a[0] = 0.0; a[1] = 0.0; a[2] = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) a[3 + i] = gq[i];
#pragma unroll
    for (int i = 0; i < 6; ++i) a[7 + i] = gnu[i];
}

template <typename T> __device__ __forceinline__ void quat_renorm(T* q) {
    T n = sqrt_(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n < T(1e-12)) { q[0] = T(1); q[1] = q[2] = q[3] = T(0); }
    else { T in = rcp_nr(n); q[0] *= in; q[1] *= in; q[2] *= in; q[3] *= in; }
}

// ---------------------------------------------------------------------------------------------------------------
// double-integrator comparison model
// ---------------------------------------------------------------------------------------------------------------
// [v_dot, w_dot] = u [K_lin | K_ang]   (dense; the input is held over the step, so this is evaluated once per step)
template <typename T, int NU>
__device__ __forceinline__ void di_accel(const Consts<T>& c, const T* __restrict__ u, T* __restrict__ acc) {
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        T s = T(0);
#pragma unroll
        for (int i = 0; i < NU; ++i) s += c.alloc[r][i] * u[i];
        acc[r] = s;
    }
}
// _di_rhs (training/train_tank_brov2_rk4.py:461-496): pos_dot = R_b2n(phi,theta,psi) v, ang_dot = w.
template <typename T>
__device__ __forceinline__ void rhs_di12(const T* __restrict__ x, const Trig<T>& tr, const T* __restrict__ acc,
                                         T* __restrict__ xd) {
    const T* nu = x + 6;
    T v1 = tr.cphi * nu[1] - tr.sphi * nu[2];
    T w1 = tr.sphi * nu[1] + tr.cphi * nu[2];
    T u2 = tr.cth * nu[0] + tr.sth * w1;
    xd[2] = tr.cth * w1 - tr.sth * nu[0];
    xd[0] = tr.cpsi * u2 - tr.spsi * v1;
    xd[1] = tr.spsi * u2 + tr.cpsi * v1;
#pragma unroll
    for (int i = 0; i < 3; ++i) xd[3 + i] = nu[3 + i];
#pragma unroll
    for (int i = 0; i < 6; ++i) xd[6 + i] = acc[i];
}
// quaternion twin (training/train_tank_brov2_wrench_quat.py:324-373): pos_dot = R(q) v, q_dot = 1/2 q (x) [0, w]
// with q normalised first.
template <typename T>
__device__ __forceinline__ void rhs_diq13(const T* __restrict__ x, const T* __restrict__ acc, T* __restrict__ xd) {
    T q[4] = {x[3], x[4], x[5], x[6]};
    quat_renorm<T>(q);
    const T qw = q[0], qx = q[1], qy = q[2], qz = q[3];
    const T* nu = x + 7;
    T R00 = T(1) - T(2) * (qy * qy + qz * qz), R01 = T(2) * (qx * qy - qz * qw), R02 = T(2) * (qx * qz + qy * qw);
    T R10 = T(2) * (qx * qy + qz * qw), R11 = T(1) - T(2) * (qx * qx + qz * qz), R12 = T(2) * (qy * qz - qx * qw);
    T R20 = T(2) * (qx * qz - qy * qw), R21 = T(2) * (qy * qz + qx * qw), R22 = T(1) - T(2) * (qx * qx + qy * qy);
    xd[0] = R00 * nu[0] + R01 * nu[1] + R02 * nu[2];
    xd[1] = R10 * nu[0] + R11 * nu[1] + R12 * nu[2];
    xd[2] = R20 * nu[0] + R21 * nu[1] + R22 * nu[2];
    const T wp = nu[3], wq = nu[4], wr = nu[5];
    xd[3] = T(0.5) * (-qx * wp - qy * wq - qz * wr);
    xd[4] = T(0.5) * (qw * wp + qy * wr - qz * wq);
    xd[5] = T(0.5) * (qw * wq - qx * wr + qz * wp);
    xd[6] = T(0.5) * (qw * wr + qx * wq - qy * wp);
#pragma unroll
    for (int i = 0; i < 6; ++i) xd[7 + i] = acc[i];
}

// ---------------------------------------------------------------------------------------------------------------
// 3rd-order thruster lag, closed form over the sub-steps of one integrator step (input held).
//
// LAGW = false: thruster coordinates, lag[8][3] = ThrusterLag._x of each thruster (the reference's hidden state).
//     y_i = G_j . lag_i + H_j F_i ; tau = alloc y                                   (128 + 124 ops per RK4 step)
//     Used by the single-evaluation kernels (rhs_kernel, thruster_wrench_kernel, thruster_series_kernel).
// LAGW = true : allocation-projected coordinates Z[6][3] = sum_i alloc[c][i] lag_i.  The eight lags are copies of ONE
//     linear filter, so any fixed linear combination of their states obeys the same recurrence driven by the same
//     combination of the inputs: tau_c = G_j . Z_c + H_j (alloc F)_c ; Z_c <- A Z_c + B (alloc F)_c.   (31 + 96 ops)
//     Identical dynamics (rounding differs at 1e-16), 18 instead of 24 hidden values.  Every rollout and evaluator
//     kernel integrates in this form; per-thruster states, when the caller wants them back, come from
//     lag_tail_kernel (brov_kernels.cuh), which replays the tail of the input history the filter still remembers.
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void allocate_wrench(const Consts<T>& c, const T* __restrict__ y, T* __restrict__ tau) {
    // rows 0..2 and 5 of the allocation matrix are structurally sparse (horizontal thrusters have no z component,
    // vertical ones only z); their zero entries are skipped at compile time (brov_set_allocation enforces them).
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        T s = T(0);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const bool nz = (r < 2) ? (i < 4) : (r == 2) ? (i >= 4) : (r == 5) ? (i < 4) : true;
            if (nz) s += c.alloc[r][i] * y[i];
        }
        tau[r] = s;
    }
}

template <typename T, bool LAGW>
__device__ __forceinline__ void thruster_tau(const Consts<T>& c, int j, const T* __restrict__ lag,
                                             const T* __restrict__ F, T* __restrict__ tau) {
    if constexpr (LAGW) {  // F holds alloc*F (6 values)
#pragma unroll
        for (int r = 0; r < 6; ++r)
            tau[r] = c.lagG[j][0] * lag[3 * r] + c.lagG[j][1] * lag[3 * r + 1] + c.lagG[j][2] * lag[3 * r + 2] +
                     c.lagH[j] * F[r];
    } else {
        T y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
            y[i] = c.lagG[j][0] * lag[3 * i] + c.lagG[j][1] * lag[3 * i + 1] + c.lagG[j][2] * lag[3 * i + 2] +
                   c.lagH[j] * F[i];
        allocate_wrench<T>(c, y, tau);
    }
}

// one filter: x <- lagA x + lagB F
template <typename T>
__device__ __forceinline__ void lag_advance1(const Consts<T>& c, T* __restrict__ x, T F) {
    const T a = x[0], b = x[1], d = x[2];
    x[0] = c.lagA[0][0] * a + c.lagA[0][1] * b + c.lagA[0][2] * d + c.lagB[0] * F;
    x[1] = c.lagA[1][0] * a + c.lagA[1][1] * b + c.lagA[1][2] * d + c.lagB[1] * F;
    x[2] = c.lagA[2][0] * a + c.lagA[2][1] * b + c.lagA[2][2] * d + c.lagB[2] * F;
}
template <typename T, bool LAGW>
__device__ __forceinline__ void lag_advance(const Consts<T>& c, T* __restrict__ lag, const T* __restrict__ F) {
#pragma unroll
    for (int i = 0; i < (LAGW ? 6 : 8); ++i) lag_advance1<T>(c, lag + 3 * i, F[i]);
}

// thruster-coordinate lag state -> allocation-projected state Z[6][3]
template <typename T>
__device__ __forceinline__ void project_lag(const Consts<T>& c, const T* __restrict__ lag24, T* __restrict__ Z) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        T y[8], t[6];
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] = lag24[3 * i + k];
        allocate_wrench<T>(c, y, t);
#pragma unroll
        for (int r = 0; r < 6; ++r) Z[3 * r + k] = t[r];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// one right-hand-side evaluation
//   lag     THRUSTER8: lag state, 8x3 (LAGW = false) or 6x3 (LAGW = true);
//           wrench models with LAG1: the 6 filtered wrench components
//   Fu      THRUSTER8 -> static thrust F[8] of this step (alloc*F[6] when LAGW); wrench models -> commanded wrench;
//           double-integrator models -> accelerations
// ---------------------------------------------------------------------------------------------------------------
// CU = false: built for "no ocean current" — the relative-velocity block and its (uniform) branch are not in the code at
// all.  The branch alone, four times per step, costs the rollout kernels 1-4 % (r02t batch 6).  (The rollout kernel's
// CU = false build also fixes the input layout at compile time, brov_kernels.cuh.)
template <typename T, int MODEL, bool LAG1, bool LAGW, class P, bool CU = true>
__device__ __forceinline__ void model_rhs(const Consts<T>& c, const P& p, int substep, const T* __restrict__ x,
                                          const Trig<T>& tr, const T* __restrict__ lag, const T* __restrict__ Fu,
                                          T* __restrict__ xd, T* __restrict__ lagd) {
    if constexpr (MODEL == MODEL_THRUSTER8) {
        T tau[6];
        thruster_tau<T, LAGW>(c, substep, lag, Fu, tau);
        rhs_euler12<T>(x, tr, tau, p, CU && c.has_current != 0, xd);
    } else if constexpr (MODEL == MODEL_DIQ13_U6) {
        rhs_diq13<T>(x, Fu, xd);
    } else if constexpr (ModelDim<MODEL>::DI) {
        rhs_di12<T>(x, tr, Fu, xd);
    } else {
        T tl[6];
        const T* tau = Fu;
        if constexpr (LAG1) {
            const T il = p[KP_ILAG1];
#pragma unroll
            for (int i = 0; i < 6; ++i) { tl[i] = lag[i]; lagd[i] = (Fu[i] - tl[i]) * il; }
            tau = tl;
        }
        if constexpr (MODEL == MODEL_WRENCH12) rhs_euler12<T>(x, tr, tau, p, CU && c.has_current != 0, xd);
        else rhs_quat13<T>(x, tau, p, CU && c.has_current != 0, xd);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// counter-based input generator: the reference's "random thrust" command signal
//     u_k = clip(0.98 u_{k-1} + 0.02 N(0,1), -1, 1)        training/train_sim_brov2_koopmanEDMDc.py:161-164,180
// generated inside the kernels instead of being streamed from HBM.  The normal deviates of (vehicle, step) come from
// Philox4x32-10 (Salmon et al., SC'11) keyed on the seed with the counter (vehicle lo, vehicle hi, step lo,
// step hi << 1 | block): any step of any vehicle can be regenerated independently, chunked / sliced / sharded rollouts
// see the identical stream.  The AR(1) state is the only thing carried (NU values per vehicle).
// ---------------------------------------------------------------------------------------------------------------
constexpr int BROV_PHILOX_ROUNDS = 10;   // the standard safety margin; 7 rounds measured 4 % faster in fp32 only
// rounds [r0, r1) of Philox4x32 on the counter block c[4]; the round keys are key + r * Weyl constants
__device__ __forceinline__ void philox_rounds(uint32_t* __restrict__ c, uint32_t k0, uint32_t k1, int r0, int r1) {
#pragma unroll
    for (int r = r0; r < r1; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        c[0] = hi1 ^ c[1] ^ (k0 + (uint32_t)r * 0x9E3779B9u);
        c[1] = lo1;
        c[2] = hi0 ^ c[3] ^ (k1 + (uint32_t)r * 0xBB67AE85u);
        c[3] = lo0;
    }
}
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t* __restrict__ out) {
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    philox_rounds(out, k0, k1, 0, BROV_PHILOX_ROUNDS);
}

// two N(0,1) deviates from two 32-bit words: Box-Muller on 23-bit uniforms, fast-math transcendentals (MUFU).
// u1 in (0, 1), u2 in [0, 1): n0 = sqrt(-2 ln u1) cos(2 pi u2), n1 = sqrt(-2 ln u1) sin(2 pi u2); |n| < 5.7.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float* __restrict__ n0, float* __restrict__ n1) {
    const float f1 = __uint_as_float(0x3f800000u | (a >> 9));            // [1, 2)
    const float f2 = __uint_as_float(0x3f800000u | (b >> 9));
    const float u1 = f1 - 0.99999994f;                                    // (0, 1]: never 0
    const float th = fmaf(f2, 6.2831855f, -6.2831855f);                   // 2 pi (f2 - 1)
    float r;                                                              // sqrt(-2 ln u1), ln = ln2 * log2
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862944f * __log2f(u1)));
    float s, c;
    __sincosf(th, &s, &c);
    *n0 = r * c;
    *n1 = r * s;
}

// The AR(1) recursion runs in float32 whatever the engine's scalar type: the command signal is a sequence of
// float32-representable numbers (half the registers in the fp64 kernels, and fp32 and fp64 engines fed the same seed
// integrate the IDENTICAL inputs); the state arrays in memory have the engine's scalar type and convert exactly.
template <typename T> struct InputGen {
    float rho;
    float sigma[8];       // sigma * scale_j
    float clip[8];        // clip * scale_j
    unsigned long long vehicle0;   // global index of local vehicle 0
    uint32_t k0, k1;      // seed
    const T* state_in;    // [n][NU] or nullptr (zeros)
    T* state_out;         // [n][NU] or nullptr
    int on;
};

// the 8 standard-normal deviates of (vehicle, step): depends on the counters only, never on the signal's state, so the
// kernels draw the deviates of step k+1 while step k integrates (integer / MUFU work under the FP pipes' latency)
template <typename T>
__device__ __forceinline__ void gen_normals(const InputGen<T>& g, unsigned long long veh, long long step,
                                            float* __restrict__ n) {
    const uint32_t v0 = (uint32_t)veh, v1 = (uint32_t)(veh >> 32);
    const uint32_t s0 = (uint32_t)step, s1 = (uint32_t)((unsigned long long)step >> 32) << 1;
    uint32_t w[8];
    philox4x32_10(v0, v1, s0, s1, g.k0, g.k1, w);
    philox4x32_10(v0, v1, s0, s1 | 1u, g.k0, g.k1, w + 4);
#pragma unroll
    for (int j = 0; j < 8; j += 2) box_muller(w[j], w[j + 1], &n[j], &n[j + 1]);
}
// s <- clip(rho s + sigma n, -clip, clip)
template <typename T, int NU>
__device__ __forceinline__ void gen_apply(const InputGen<T>& g, const float* __restrict__ n, float* __restrict__ s) {
#pragma unroll
    for (int j = 0; j < NU; ++j) s[j] = fminf(fmaxf(fmaf(g.rho, s[j], g.sigma[j] * n[j]), -g.clip[j]), g.clip[j]);
}
// advance the AR(1) input state s[NU] of global vehicle `veh` to global step `step`
template <typename T, int NU>
__device__ __forceinline__ void gen_advance(const InputGen<T>& g, unsigned long long veh, long long step,
                                            float* __restrict__ s) {
    float n[8];
    gen_normals<T>(g, veh, step, n);
    gen_apply<T, NU>(g, n, s);
}

// The command signal of the NEXT step, produced in slices between the stages of the current step (integrate_step
// calls work(0..3)): the Philox rounds are dependent integer multiplies and the Box-Muller transform is MUFU work —
// placed in one lump at the top of the step they stall a warp that has only one other warp to hide behind (fp64: +30 %
// per step measured, r02f); spread through the step they issue into the latency gaps of the FP pipes.  One counter
// block (4 words -> 4 deviates -> 4 channels) at a time; the AR(1) state gs[] is advanced in place as soon as a block
// is done — the current step converted it to inputs before its first stage and does not look at it again.
template <typename T, int NU> struct GenSide {
    const InputGen<T>& g;
    float* gs;            // AR(1) state, NU channels: on entry to a step the state that step uses
    uint32_t c[4];        // counter block in flight
    uint32_t v0, v1, s0, s1;
    bool advance;         // false on the last step of a launch: the state handed on is the last one USED
    __device__ __forceinline__ GenSide(const InputGen<T>& g_, float* gs_) : g(g_), gs(gs_), advance(true) {}
    __device__ __forceinline__ void start(unsigned long long veh, long long step, bool adv) {
        v0 = (uint32_t)veh; v1 = (uint32_t)(veh >> 32);
        s0 = (uint32_t)step; s1 = (uint32_t)((unsigned long long)step >> 32) << 1;
        advance = adv;
    }
    __device__ __forceinline__ void block(int b) { c[0] = v0; c[1] = v1; c[2] = s0; c[3] = s1 | (uint32_t)b; }
    __device__ __forceinline__ void finish(int b) {
        float n[4];
        box_muller(c[0], c[1], &n[0], &n[1]);
        box_muller(c[2], c[3], &n[2], &n[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int q = 4 * b + j;
            if (q < NU) {
                const float v = fminf(fmaxf(fmaf(g.rho, gs[q], g.sigma[q] * n[j]), -g.clip[q]), g.clip[q]);
                gs[q] = advance ? v : gs[q];
            }
        }
    }
    // slice s of 4 (RK4: one per stage); all(): everything at once (Euler step, prologue)
    __device__ __forceinline__ void work(int s) {
        constexpr int R = BROV_PHILOX_ROUNDS;
        if (s == 0) { block(0); philox_rounds(c, g.k0, g.k1, 0, R / 2); }
        else if (s == 1) { philox_rounds(c, g.k0, g.k1, R / 2, R); finish(0); }
        else if (s == 2) { block(1); philox_rounds(c, g.k0, g.k1, 0, R / 2); }
        else { philox_rounds(c, g.k0, g.k1, R / 2, R); finish(1); }
    }
    __device__ __forceinline__ void all() { work(0); work(1); work(2); work(3); }
};
// register prefetch of the NEXT step's command row issued between the stages of the current one: before stage 3 the
// row's registers are live for half a step instead of a whole one (measured r02t, fp64 thruster rollout per 1000
// steps: at the top of the step 4.28 ms, before stage 2 4.33, before stage 3 4.12, before stage 4 4.19)
template <class F> struct LateSide {
    F f;
    int at;
    __device__ __forceinline__ void work(int s) { if (s == at) f(); }
    __device__ __forceinline__ void all() { f(); }
};
struct NoSide {
    __device__ __forceinline__ NoSide() {}
    template <class G> __device__ __forceinline__ NoSide(const G&, float*) {}
    __device__ __forceinline__ void work(int) {}
    __device__ __forceinline__ void all() {}
};

// ---------------------------------------------------------------------------------------------------------------
// one integrator step of one vehicle (the body of simulate_physics' loop: RK4 training/train_tank_brov2_rk4.py:386-394,
// Euler training/train_tank_brov2_full_comparison.py:462-465, quaternion re-normalisation
// training/train_tank_brov2_wrench_quat.py:262-263)
//   x[NX]   state (registers, in/out)
//   lag     THRUSTER8: allocation-projected lag state Z[6][3]; wrench models with LAG1: filtered wrench [6]
//   u[NU]   input held over the step
//   abs_cth |cos theta| of the state the step starts from (Euler-angle Fossen models; 1 otherwise): how close the
//           vehicle is to the singularity of the Euler-rate kinematics (fossen/BlueROV2.py:43-62)
// ---------------------------------------------------------------------------------------------------------------
//   side    work to interleave with the step (GenSide: the next step's input deviates; NoSide: nothing)
template <typename T, int MODEL, int INTEG, bool LAG1, class P, class SIDE, bool CU = true>
__device__ __forceinline__ void integrate_step(const Consts<T>& c, const P& p, T* __restrict__ x, T* __restrict__ lag,
                                               const T* __restrict__ u, T& abs_cth, SIDE& side) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr int NL = LAG1 ? 6 : 1;  // continuous auxiliary states integrated with x
    constexpr bool LAGW = true;
    const T dt = c.dt;
    T Fu[ModelDim<MODEL>::NU];
    if constexpr (MODEL == MODEL_THRUSTER8) {
        T F[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) F[i] = thrust_poly<T>(c, u[i]);
        allocate_wrench<T>(c, F, Fu);
    } else if constexpr (ModelDim<MODEL>::DI) {
        di_accel<T, ModelDim<MODEL>::NU>(c, u, Fu);
        // the quaternion twin normalises the stored quaternion BEFORE the step (wrench_quat.py:345)
        if constexpr (MODEL == MODEL_DIQ13_U6) quat_renorm<T>(x + 3);
    } else {
#pragma unroll
        for (int i = 0; i < 6; ++i) Fu[i] = u[i];
    }
    T k[NX], kl[NL];
    constexpr bool EULER_ANGLES = !ModelDim<MODEL>::QUAT;
    Trig<T> tr0;
    if constexpr (EULER_ANGLES) trig_full<T>(c, x + 3, tr0);
    abs_cth = (EULER_ANGLES && !ModelDim<MODEL>::DI) ? abs_(tr0.cth) : T(1);
    if constexpr (INTEG == INTEG_EULER) {
        model_rhs<T, MODEL, LAG1, LAGW, P, CU>(c, p, 0, x, tr0, lag, Fu, k, kl);
        side.all();
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt * k[i];
        if constexpr (LAG1) {
#pragma unroll
            for (int i = 0; i < 6; ++i) lag[i] += dt * kl[i];
        }
    } else {
        // classic RK4 in low-storage form: acc accumulates k1 + 2 k2 + 2 k3 + k4, xs is the stage state
        T acc[NX], xs[NX], accl[NL], ls[NL];
        const T hdt = T(0.5) * dt;
        Trig<T> trs;
        T dang[3];
        model_rhs<T, MODEL, LAG1, LAGW, P, CU>(c, p, 0, x, tr0, lag, Fu, k, kl);
#pragma unroll
        for (int s = 1; s <= 3; ++s) {
            side.work(s - 1);
            const T w = (s == 1) ? T(1) : T(2);   // weight of the stage just evaluated
            const T h = (s == 3) ? dt : hdt;      // offset of the next stage
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                if (s == 1) acc[i] = k[i]; else acc[i] += w * k[i];
                xs[i] = x[i] + h * k[i];
            }
            if constexpr (LAG1) {
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    if (s == 1) accl[i] = kl[i]; else accl[i] += w * kl[i];
                    ls[i] = lag[i] + h * kl[i];
                }
            }
            if constexpr (EULER_ANGLES) {
#pragma unroll
                for (int i = 0; i < 3; ++i) dang[i] = h * k[3 + i];
                trig_stage(c, tr0, dang, xs + 3, trs);
            }
            model_rhs<T, MODEL, LAG1, LAGW, P, CU>(c, p, s, xs, trs, LAG1 ? ls : lag, Fu, k, kl);
        }
        side.work(3);
        const T dt6 = dt * T(1.0 / 6.0);
#pragma unroll
        for (int i = 0; i < NX; ++i) x[i] += dt6 * (acc[i] + k[i]);
        if constexpr (LAG1) {
#pragma unroll
            for (int i = 0; i < 6; ++i) lag[i] += dt6 * (accl[i] + kl[i]);
        }
    }
    if constexpr (MODEL == MODEL_THRUSTER8) lag_advance<T, LAGW>(c, lag, Fu);
    if constexpr (ModelDim<MODEL>::QUAT) quat_renorm<T>(x + 3);
}

// ---------------------------------------------------------------------------------------------------------------
// forward-mode sensitivities: a dual number (value, tangent), both fp64.  nu_dot, rhs_euler12, rhs_quat13 and
// quat_renorm instantiated with it carry the derivative of the state along one direction of the coefficient vector
// (brov_grad.cu).  The derivative is that of the function the code computes, branch taken: d|x| = sign(x) dx with
// sign(0) = 0, the clamped cos(theta) and the quaternion fallback are constants.  Comparisons look at the value.
// ---------------------------------------------------------------------------------------------------------------
struct Dual {
    double v, d;
    Dual() = default;
    __device__ __forceinline__ Dual(double x) : v(x), d(0.0) {}
    __device__ __forceinline__ Dual(double x, double dx) : v(x), d(dx) {}
};
__device__ __forceinline__ Dual operator+(Dual a, Dual b) { return Dual(a.v + b.v, a.d + b.d); }
__device__ __forceinline__ Dual operator-(Dual a, Dual b) { return Dual(a.v - b.v, a.d - b.d); }
__device__ __forceinline__ Dual operator-(Dual a) { return Dual(-a.v, -a.d); }
__device__ __forceinline__ Dual operator*(Dual a, Dual b) { return Dual(a.v * b.v, fma(a.v, b.d, a.d * b.v)); }
__device__ __forceinline__ Dual operator*(double a, Dual b) { return Dual(a * b.v, a * b.d); }
__device__ __forceinline__ Dual operator*(Dual a, double b) { return Dual(a.v * b, a.d * b); }
__device__ __forceinline__ Dual& operator+=(Dual& a, Dual b) { a = a + b; return a; }
__device__ __forceinline__ Dual& operator-=(Dual& a, Dual b) { a = a - b; return a; }
__device__ __forceinline__ Dual& operator*=(Dual& a, Dual b) { a = a * b; return a; }
__device__ __forceinline__ bool operator<(Dual a, Dual b) { return a.v < b.v; }
__device__ __forceinline__ bool operator>(Dual a, Dual b) { return a.v > b.v; }
__device__ __forceinline__ bool operator==(Dual a, Dual b) { return a.v == b.v; }
__device__ __forceinline__ Dual abs_(Dual a) {
    const double s = a.v > 0.0 ? 1.0 : (a.v < 0.0 ? -1.0 : 0.0);
    return Dual(fabs(a.v), s * a.d);
}
__device__ __forceinline__ Dual sqrt_(Dual a) {
    const double r = sqrt(a.v);
    return Dual(r, 0.5 * a.d * rcp_nr(r));
}
__device__ __forceinline__ Dual rcp_nr(Dual a) {
    const double r = rcp_nr(a.v);
    return Dual(r, -a.d * r * r);
}
__device__ __forceinline__ void sincos_(Dual a, Dual* s, Dual* c, const double* K = kSinCos64) {
    double sv, cv;
    sincos_(a.v, &sv, &cv, K);
    *s = Dual(sv, cv * a.d);
    *c = Dual(cv, -sv * a.d);
}

// kernel coefficients of a dual evaluation: the point kp (shared by the block) with the tangent dk of this thread's
// direction
struct ParamsDual {
    const double* kp;
    const double* dk;
    __device__ __forceinline__ Dual operator[](int i) const { return Dual(kp[i], dk[i]); }
};

// integrate_step with the state carried as dual numbers.  The thruster map, the T200 polynomial and the lag do not
// depend on the coefficients: they stay plain double and the body wrench enters the dual right-hand side as a
// constant.  Every stage evaluates its sines and cosines in full (no stage-rotation shortcut), so the values agree
// with integrate_step to rounding, not bit for bit.
template <int MODEL, int INTEG, class P>
__device__ __forceinline__ void integrate_step_dual(const Consts<double>& c, const P& p, Dual* __restrict__ x,
                                                    double* __restrict__ lag, const double* __restrict__ u,
                                                    double& abs_cth) {
    constexpr int NX = ModelDim<MODEL>::NX;
    constexpr bool EULER_ANGLES = !ModelDim<MODEL>::QUAT;
    const bool cur = c.has_current != 0;
    const double dt = c.dt;
    double Fu[6];
    if constexpr (MODEL == MODEL_THRUSTER8) {
        double F[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) F[i] = thrust_poly<double>(c, u[i]);
        allocate_wrench<double>(c, F, Fu);
    } else {
#pragma unroll
        for (int i = 0; i < 6; ++i) Fu[i] = u[i];
    }
    auto rhs = [&](int s, const Dual* xs, Dual* out) {
        Dual tau[6];
        if constexpr (MODEL == MODEL_THRUSTER8) {
            double t[6];
            thruster_tau<double, true>(c, s, lag, Fu, t);
#pragma unroll
            for (int r = 0; r < 6; ++r) tau[r] = Dual(t[r]);
        } else {
#pragma unroll
            for (int r = 0; r < 6; ++r) tau[r] = Dual(Fu[r]);
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
    if constexpr (MODEL == MODEL_THRUSTER8) lag_advance<double, true>(c, lag, Fu);
    if constexpr (ModelDim<MODEL>::QUAT) quat_renorm<Dual>(x + 3);
}

}  // namespace brov
