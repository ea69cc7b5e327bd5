// brov_api.cu — the C ABI of libbrov.so (include/brov.h): engine handle, host-side constant preparation in extended
// precision (mass matrix inverse, Coriolis coefficient differences, thruster allocation from the reference's
// geometry formula, zero-order-hold discretisation of the thruster lag and its closed form over the sub-steps of an
// integrator step), argument validation, kernel launches, and the host-buffer streaming rollout.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <type_traits>
#include <vector>

#include "../../include/brov.h"
#include "brov_internal.cuh"
#include "brov_kernels.cuh"
#include "brov_grad.cuh"
#include "brov_lin.cuh"
#include "brov_cl.cuh"
#include "brov_adj.cuh"

using namespace brov;

static_assert(BROV_NKP == KP_COUNT, "coefficient vector length");
static_assert(BROV_MAX_H == MAX_H, "horizon count");

// ---------------------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int brov::fail_msg(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) return fail(BROV_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

extern "C" const char* brov_last_error(void) { return g_err; }
extern "C" int brov_abi_version(void) { return BROV_ABI_VERSION; }

// ---------------------------------------------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------------------------------------------
struct LagDisc {
    double dt;
    double Ad[9];
    double Bd[3];
};

struct HostStage {  // resources of brov_rollout_host, grown on demand
    void* d_x = nullptr;
    void* d_lag = nullptr;       // carried between chunks: allocation-projected [n][18] (thruster model) / [n][6]
    void* d_lag24 = nullptr;     // per-thruster states [n][24]: caller's lag_in, then the rebuilt lag_out
    void* d_gen = nullptr;       // AR(1) state of generated inputs [n][NU]
    void* d_health = nullptr;    // unsigned long long[2] + per-vehicle running min |cos theta| [n]
    size_t cap_lag24 = 0, cap_gen = 0, cap_health = 0;
    void* d_u[2] = {nullptr, nullptr};
    void* d_traj[2] = {nullptr, nullptr};
    size_t cap_x = 0, cap_lag = 0, cap_u = 0, cap_traj = 0;
    cudaStream_t s_compute = nullptr, s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    bool ready = false;
};

struct brov_engine {
    int model, dtype, device;
    double kp[KP_COUNT];
    double alloc[6][8];
    int use_lag1;
    const void* pv;
    long long pv_n;
    int pv_current;      // some row of the per-vehicle table has a non-zero current (relative-velocity terms needed)
    std::vector<LagDisc> lag_overrides;
    LagDisc lag_cache;
    HostStage hs;
    int num_sms;
    int* d_sched;        // [1 + nvblocks] ticket counter + per-vehicle-block progress flags (temporal tiling)
    size_t cap_sched;    // in ints
    // engine-owned scratch of brov_rollout (grown on demand): hand-over of the lag / generator state between time slices
    // when the caller passes no buffer of the right shape, running min |cos theta| for the health counters, and the
    // generator state snapshot the per-thruster lag epilogue restarts from
    void* d_scratch[4];
    size_t cap_scratch[4];
    // staging of the host-buffer single-call entry points (brov_rhs_host, brov_thruster_wrench_host)
    void* call_pinned;   // pinned host buffer
    void* call_dev;      // device mirror
    size_t cap_call;     // bytes of each
    cudaStream_t call_stream;
};

static const double LAG_AC[9] = {-89.0, -72.33, -26.54, 128.0, 0.0, 0.0, 0.0, 32.0, 0.0};  // fossen/BlueROV2.py:476-478
static const double LAG_BC[3] = {8.0, 0.0, 0.0};                                             // :479
static const double LAG_CC[3] = {0.0, 5.992, 3.317};                                         // :480

static int model_nx(int m) { return (m == BROV_WRENCH_QUAT13 || m == BROV_DI_QUAT13_U6) ? 13 : 12; }
static int model_nu(int m) { return (m == BROV_THRUSTER8_LAG3 || m == BROV_DI_EULER12_U8) ? 8 : 6; }
// the state z of the linearize, EKF, closed-loop and adjoint calls: x and, thruster8, the 18 projected lag states
static int model_nz(int m) { return model_nx(m) + (m == BROV_THRUSTER8_LAG3 ? 18 : 0); }
static bool model_is_di(int m) { return m >= BROV_DI_EULER12_U8 && m <= BROV_DI_QUAT13_U6; }
static int model_nlag(const brov_engine* e) {
    return e->model == BROV_THRUSTER8_LAG3 ? 24 : (e->use_lag1 ? 6 : 0);
}
static size_t scalar_size(int dtype) { return dtype == BROV_F32 ? 4 : 8; }

// ---------------------------------------------------------------------------------------------------------------
// constants
// ---------------------------------------------------------------------------------------------------------------
extern "C" int brov_default_physical(double rho, double* ph) {
    if (!ph) return fail(BROV_EINVAL, "phys is NULL");
    const double g = 9.82, m = 13.5, vol = 0.0134;
    ph[BROV_PH_M] = m;
    ph[BROV_PH_W] = m * g;
    ph[BROV_PH_B] = rho * g * vol;
    ph[BROV_PH_XB + 0] = 0.0; ph[BROV_PH_XB + 1] = 0.0; ph[BROV_PH_XB + 2] = -0.01;
    ph[BROV_PH_I + 0] = 0.26; ph[BROV_PH_I + 1] = 0.23; ph[BROV_PH_I + 2] = 0.37;
    const double added[6] = {-6.36, -7.12, -18.68, -0.189, -0.135, -0.222};
    const double lin[6] = {-13.7, -0.0, -33.0, -0.0, -0.8, -0.0};
    const double quad[6] = {-141.0, -217.0, -190.0, -1.19, -0.47, -1.5};
    for (int i = 0; i < 6; ++i) {
        ph[BROV_PH_ADDED + i] = added[i];
        ph[BROV_PH_LIN + i] = lin[i];
        ph[BROV_PH_QUAD + i] = quad[i];
    }
    for (int i = 0; i < 3; ++i) {
        ph[BROV_PH_MINV + i] = 1.0 / (m - added[i]);
        ph[BROV_PH_MINV + 3 + i] = 1.0 / (ph[BROV_PH_I + i] - added[3 + i]);
        ph[BROV_PH_CURRENT + i] = 0.0;
    }
    ph[BROV_PH_TLAG1] = 0.0;
    return BROV_OK;
}

extern "C" int brov_derive_params(const double* ph, double* kp) {
    if (!ph || !kp) return fail(BROV_EINVAL, "NULL argument");
    const double m = ph[BROV_PH_M];
    double a[3], b[3];
    for (int i = 0; i < 3; ++i) {
        a[i] = m - ph[BROV_PH_ADDED + i];
        b[i] = ph[BROV_PH_I + i] - ph[BROV_PH_ADDED + 3 + i];
    }
    for (int i = 0; i < 6; ++i) kp[KP_MINV + i] = ph[BROV_PH_MINV + i];
    for (int i = 0; i < 3; ++i) kp[KP_A + i] = a[i];
    kp[KP_DA + 0] = a[2] - a[1]; kp[KP_DA + 1] = a[0] - a[2]; kp[KP_DA + 2] = a[1] - a[0];
    kp[KP_DB + 0] = b[2] - b[1]; kp[KP_DB + 1] = b[0] - b[2]; kp[KP_DB + 2] = b[1] - b[0];
    for (int i = 0; i < 6; ++i) {
        kp[KP_DL + i] = -ph[BROV_PH_LIN + i];
        kp[KP_DQ + i] = -ph[BROV_PH_QUAD + i];
    }
    kp[KP_WMB] = ph[BROV_PH_W] - ph[BROV_PH_B];
    for (int i = 0; i < 3; ++i) {
        kp[KP_XBB + i] = ph[BROV_PH_XB + i] * ph[BROV_PH_B];
        kp[KP_CUR + i] = ph[BROV_PH_CURRENT + i];
    }
    kp[KP_ILAG1] = ph[BROV_PH_TLAG1] > 0.0 ? 1.0 / ph[BROV_PH_TLAG1] : 0.0;
    kp[KP_ILAG1 + 1] = 0.0;
    return BROV_OK;
}

// Thruster geometry: r_i = Rz(alpha_i) r_base, e_i = Rz(beta_i) e_base with the paper's rounded placement angles
// (fossen/BlueROV2.py:172-232; never symmetrised, SURVEY trap T6); column i of the allocation is [e_i; r_i x e_i].
extern "C" int brov_default_allocation(double* alloc, double* r_out, double* dir_out) {
    const double PI = 3.141592653589793;
    const double r_h[3] = {0.156, 0.111, 0.085}, r_v[3] = {0.12, 0.218, 0.0};
    const double s2 = 1.0 / std::sqrt(2.0);
    const double e_h[3] = {s2, -s2, 0.0};
    const double ang_r[8] = {0.0, 5.05, 1.91, PI, 0.0, 4.15, 1.01, PI};
    const double ang_e[4] = {0.0, PI / 2, 3 * PI / 2, PI};
    for (int i = 0; i < 8; ++i) {
        const double* rb = i < 4 ? r_h : r_v;
        double c = std::cos(ang_r[i]), s = std::sin(ang_r[i]);
        double r[3] = {c * rb[0] - s * rb[1], s * rb[0] + c * rb[1], rb[2]};
        double e[3];
        if (i < 4) {
            double ce = std::cos(ang_e[i]), se = std::sin(ang_e[i]);
            e[0] = ce * e_h[0] - se * e_h[1];
            e[1] = se * e_h[0] + ce * e_h[1];
            e[2] = e_h[2];
        } else {
            e[0] = 0.0; e[1] = 0.0; e[2] = -1.0;
        }
        if (alloc) {
            alloc[0 * 8 + i] = e[0];
            alloc[1 * 8 + i] = e[1];
            alloc[2 * 8 + i] = e[2];
            alloc[3 * 8 + i] = r[1] * e[2] - r[2] * e[1];
            alloc[4 * 8 + i] = r[2] * e[0] - r[0] * e[2];
            alloc[5 * 8 + i] = r[0] * e[1] - r[1] * e[0];
        }
        for (int j = 0; j < 3; ++j) {
            if (r_out) r_out[3 * i + j] = r[j];
            if (dir_out) dir_out[3 * i + j] = e[j];
        }
    }
    return BROV_OK;
}

// exp([[A, B], [0, 0]] dt) by scaling and squaring of a Taylor series in long double: (Ad, Bd) of the zero-order hold,
// i.e. what scipy.signal.cont2discrete(method='zoh') returns at fossen/BlueROV2.py:494-495.
extern "C" int brov_lag_discretize(double dt, double* Ad, double* Bd) {
    if (!Ad || !Bd || !(dt > 0.0) || !std::isfinite(dt)) return fail(BROV_EINVAL, "brov_lag_discretize: bad dt or NULL output");
    typedef long double ld;
    ld M[4][4] = {{0}};
    ld nrm = 0;
    for (int i = 0; i < 3; ++i) {
        ld row = 0;
        for (int j = 0; j < 3; ++j) { M[i][j] = (ld)LAG_AC[3 * i + j] * (ld)dt; row += fabsl(M[i][j]); }
        M[i][3] = (ld)LAG_BC[i] * (ld)dt;
        row += fabsl(M[i][3]);
        if (row > nrm) nrm = row;
    }
    int s = 0;
    while (nrm > 0.0625L) { nrm *= 0.5L; ++s; }
    ld scale = ldexpl(1.0L, -s);
    for (auto& row : M) for (auto& v : row) v *= scale;
    ld E[4][4], term[4][4], tmp[4][4];
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) E[i][j] = term[i][j] = (i == j) ? 1.0L : 0.0L;
    for (int k = 1; k <= 24; ++k) {
        for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) {
            ld v = 0;
            for (int q = 0; q < 4; ++q) v += term[i][q] * M[q][j];
            tmp[i][j] = v / (ld)k;
        }
        for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) { term[i][j] = tmp[i][j]; E[i][j] += tmp[i][j]; }
    }
    for (int q = 0; q < s; ++q) {
        for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) {
            ld v = 0;
            for (int r = 0; r < 4; ++r) v += E[i][r] * E[r][j];
            tmp[i][j] = v;
        }
        memcpy(E, tmp, sizeof(E));
    }
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) Ad[3 * i + j] = (double)E[i][j];
        Bd[i] = (double)E[i][3];
    }
    return BROV_OK;
}

static const LagDisc* lag_for_dt(brov_engine* e, double dt) {
    for (const auto& o : e->lag_overrides)
        if (o.dt == dt) return &o;
    if (e->lag_cache.dt != dt) {
        if (brov_lag_discretize(dt, e->lag_cache.Ad, e->lag_cache.Bd) != BROV_OK) return nullptr;
        e->lag_cache.dt = dt;
    }
    return &e->lag_cache;
}

template <typename T>
static int make_consts(brov_engine* e, double dt, int nsub, Consts<T>* c) {
    memset(c, 0, sizeof(*c));
    for (int i = 0; i < KP_COUNT; ++i) c->kp[i] = (T)e->kp[i];
    for (int r = 0; r < 6; ++r) for (int i = 0; i < 8; ++i) c->alloc[r][i] = (T)e->alloc[r][i];
    c->dt = (T)dt;
    {
        const double poly[5] = {-140.3, 389.9, -404.1, 176.0, 8.9};   // fossen/BlueROV2.py:251-257, highest power first
        const double sc[16] = {0.6366197723675814, 1.5707963267948966, 6.123233995736766e-17, -1.4973849048591698e-33,
                               -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04,
                               2.75573137070700676789e-06, -2.50507602534068634195e-08, 1.58969099521155010221e-10,
                               4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05,
                               -2.75573143513906633035e-07, 2.08757232129817482790e-09, -1.13596475577881948265e-11};
        const double rot[8] = {-1.6666666666666667e-1, 8.3333333333333333e-3, -1.9841269841269841e-4, -0.5,
                               4.1666666666666667e-2, -1.3888888888888889e-3, 2.4801587301587302e-5, 0.0};
        for (int i = 0; i < 5; ++i) c->poly[i] = (T)poly[i];
        for (int i = 0; i < 16; ++i) c->sc[i] = (T)sc[i];
        for (int i = 0; i < 8; ++i) c->rot[i] = (T)rot[i];
    }
    // per-vehicle tables: the caller says whether any row carries an ocean current (the table is device memory)
    c->has_current = (e->pv ? e->pv_current != 0
                            : (e->kp[KP_CUR] != 0.0 || e->kp[KP_CUR + 1] != 0.0 || e->kp[KP_CUR + 2] != 0.0)) ? 1 : 0;
    c->use_lag1 = e->use_lag1;
    if (e->model == BROV_THRUSTER8_LAG3) {
        const LagDisc* d = lag_for_dt(e, dt);
        if (!d) return BROV_EINVAL;
        typedef long double ld;
        ld P[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, S[3][3] = {{0}}, tmp[3][3];
        for (int j = 0; j < nsub; ++j) {
            for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) S[a][b] += P[a][b];       // S_{j+1}
            for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) {                          // P = Ad^{j+1}
                ld v = 0;
                for (int q = 0; q < 3; ++q) v += P[a][q] * (ld)d->Ad[3 * q + b];
                tmp[a][b] = v;
            }
            memcpy(P, tmp, sizeof(P));
            ld h = 0;
            for (int b = 0; b < 3; ++b) {
                ld g = 0, sb = 0;
                for (int a = 0; a < 3; ++a) g += (ld)LAG_CC[a] * P[a][b];
                c->lagG[j][b] = (T)(double)g;
                for (int q = 0; q < 3; ++q) sb += S[b][q] * (ld)d->Bd[q];
                h += (ld)LAG_CC[b] * sb;
            }
            c->lagH[j] = (T)(double)h;
        }
        for (int a = 0; a < 3; ++a) {
            ld sb = 0;
            for (int b = 0; b < 3; ++b) { c->lagA[a][b] = (T)(double)P[a][b]; sb += S[a][b] * (ld)d->Bd[b]; }
            c->lagB[a] = (T)(double)sb;
        }
    }
    return BROV_OK;
}

extern "C" int brov_create(int model, int dtype, int device, brov_engine_t** out) {
    if (!out) return fail(BROV_EINVAL, "out is NULL");
    *out = nullptr;
    if (model < 0 || model > BROV_DI_QUAT13_U6) return fail(BROV_EINVAL, "unknown model %d", model);
    if (dtype != BROV_F64 && dtype != BROV_F32) return fail(BROV_EINVAL, "unknown dtype %d", dtype);
    int ndev = 0;
    CUDA_TRY(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(BROV_EINVAL, "device %d out of range (%d visible)", device, ndev);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(BROV_EUNSUPPORTED, "libbrov is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    brov_engine* e = new (std::nothrow) brov_engine();
    if (!e) return fail(BROV_ENOMEM, "out of host memory");
    e->model = model; e->dtype = dtype; e->device = device;
    e->use_lag1 = 0; e->pv = nullptr; e->pv_n = 0; e->pv_current = 0;
    e->lag_cache.dt = -1.0;
    e->num_sms = prop.multiProcessorCount; e->d_sched = nullptr; e->cap_sched = 0;
    for (int i = 0; i < 4; ++i) { e->d_scratch[i] = nullptr; e->cap_scratch[i] = 0; }
    e->call_pinned = nullptr; e->call_dev = nullptr; e->cap_call = 0; e->call_stream = nullptr;
    double ph[BROV_NPHYS];
    brov_default_physical(1000.0, ph);
    brov_derive_params(ph, e->kp);
    brov_default_allocation(&e->alloc[0][0], nullptr, nullptr);
    if (model_is_di(model)) memset(e->alloc, 0, sizeof(e->alloc));  // gains arrive through brov_set_di_gains
    *out = e;
    return BROV_OK;
}

static void hs_release(brov_engine* e) {
    HostStage& h = e->hs;
    cudaSetDevice(e->device);
    cudaFree(h.d_x); cudaFree(h.d_lag); cudaFree(h.d_lag24); cudaFree(h.d_gen); cudaFree(h.d_health);
    for (int b = 0; b < 2; ++b) {
        cudaFree(h.d_u[b]); cudaFree(h.d_traj[b]);
        if (h.ev_in[b]) cudaEventDestroy(h.ev_in[b]);
        if (h.ev_done[b]) cudaEventDestroy(h.ev_done[b]);
        if (h.ev_out[b]) cudaEventDestroy(h.ev_out[b]);
    }
    if (h.s_compute) cudaStreamDestroy(h.s_compute);
    if (h.s_in) cudaStreamDestroy(h.s_in);
    if (h.s_out) cudaStreamDestroy(h.s_out);
    h = HostStage();
}

extern "C" void brov_destroy(brov_engine_t* e) {
    if (!e) return;
    hs_release(e);
    if (e->d_sched) cudaFree(e->d_sched);
    for (int i = 0; i < 4; ++i) if (e->d_scratch[i]) cudaFree(e->d_scratch[i]);
    if (e->call_pinned) cudaFreeHost(e->call_pinned);
    if (e->call_dev) cudaFree(e->call_dev);
    if (e->call_stream) cudaStreamDestroy(e->call_stream);
    delete e;
}

extern "C" int brov_set_params(brov_engine_t* e, const double* kp) {
    if (!e || !kp) return fail(BROV_EINVAL, "NULL argument");
    for (int i = 0; i < KP_COUNT; ++i) {
        if (!std::isfinite(kp[i])) return fail(BROV_EINVAL, "coefficient %d is not finite", i);
        e->kp[i] = kp[i];
    }
    return BROV_OK;
}
extern "C" int brov_get_params(const brov_engine_t* e, double* kp) {
    if (!e || !kp) return fail(BROV_EINVAL, "NULL argument");
    memcpy(kp, e->kp, sizeof(e->kp));
    return BROV_OK;
}
extern "C" int brov_set_di_gains(brov_engine_t* e, const double* K_lin, const double* K_ang) {
    if (!e || !K_lin || !K_ang) return fail(BROV_EINVAL, "NULL argument");
    if (!model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "brov_set_di_gains needs a BROV_DI_* engine");
    const int nu = model_nu(e->model);
    memset(e->alloc, 0, sizeof(e->alloc));
    for (int i = 0; i < nu; ++i)
        for (int r = 0; r < 3; ++r) {
            if (!std::isfinite(K_lin[i * 3 + r]) || !std::isfinite(K_ang[i * 3 + r])) return fail(BROV_EINVAL, "gain [%d][%d] is not finite", i, r);
            e->alloc[r][i] = K_lin[i * 3 + r];
            e->alloc[3 + r][i] = K_ang[i * 3 + r];
        }
    return BROV_OK;
}
extern "C" int brov_set_allocation(brov_engine_t* e, const double* alloc) {
    if (!e || !alloc) return fail(BROV_EINVAL, "NULL argument");
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "double-integrator engines take brov_set_di_gains");
    // the kernel skips the structural zeros of the BlueROV2 heavy layout (4 horizontal + 4 vertical thrusters)
    for (int r = 0; r < 6; ++r)
        for (int i = 0; i < 8; ++i) {
            const bool nz = (r < 2) ? (i < 4) : (r == 2) ? (i >= 4) : (r == 5) ? (i < 4) : true;
            if (!nz && alloc[r * 8 + i] != 0.0)
                return fail(BROV_EUNSUPPORTED, "allocation[%d][%d] must be zero (horizontal thrusters 0-3 act in x,y,N; vertical 4-7 in z)", r, i);
        }
    memcpy(e->alloc, alloc, sizeof(e->alloc));
    return BROV_OK;
}
extern "C" int brov_set_vehicle_params(brov_engine_t* e, const void* kp_soa_dev, long long n, int any_current) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (kp_soa_dev && n <= 0) return fail(BROV_EINVAL, "vehicle table with n = %lld", n);
    if (kp_soa_dev && model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "double-integrator engines have no per-vehicle coefficient table");
    e->pv = kp_soa_dev;
    e->pv_n = kp_soa_dev ? n : 0;
    e->pv_current = (kp_soa_dev && any_current) ? 1 : 0;
    return BROV_OK;
}
extern "C" int brov_set_wrench_lag1(brov_engine_t* e, int enable) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (enable && (e->model == BROV_THRUSTER8_LAG3 || model_is_di(e->model)))
        return fail(BROV_EUNSUPPORTED, "the first-order wrench lag applies to the wrench-input Fossen models only");
    e->use_lag1 = enable ? 1 : 0;
    return BROV_OK;
}
extern "C" int brov_set_lag_discrete(brov_engine_t* e, double dt, const double* Ad, const double* Bd) {
    if (!e || !Ad || !Bd) return fail(BROV_EINVAL, "NULL argument");
    LagDisc d;
    d.dt = dt;
    memcpy(d.Ad, Ad, sizeof(d.Ad));
    memcpy(d.Bd, Bd, sizeof(d.Bd));
    for (auto& o : e->lag_overrides)
        if (o.dt == dt) { o = d; return BROV_OK; }
    e->lag_overrides.push_back(d);
    return BROV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// device entry points
// ---------------------------------------------------------------------------------------------------------------
static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

template <typename T>
static int rhs_impl(brov_engine* e, long long n, const void* x, const void* u, void* lag, double dt, void* xdot, cudaStream_t st) {
    RhsArgs<T> a;
    int rc = make_consts<T>(e, dt, 1, &a.c);
    if (rc) return rc;
    a.x = (const T*)x; a.u = (const T*)u; a.lag = (T*)lag; a.pv = (const T*)e->pv; a.xdot = (T*)xdot; a.n = (int)n;
    CUDA_TRY(launch_rhs<T>(e->model, e->use_lag1 != 0, a, st));
    return BROV_OK;
}

extern "C" int brov_rhs(brov_engine_t* e, long long n, const void* x, const void* u, void* lag, double dt, void* xdot, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (n < 0 || n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", n);
    if (n == 0) return BROV_OK;
    if (!x || !u || !xdot) return fail(BROV_EINVAL, "x, u and xdot must not be NULL");
    if (e->model == BROV_THRUSTER8_LAG3 && !(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0 (it fixes the lag discretisation)");
    if (e->pv && e->pv_n != n) return fail(BROV_EINVAL, "vehicle table has %lld rows, call has n = %lld", e->pv_n, n);
    CUDA_TRY(cudaSetDevice(e->device));
    return e->dtype == BROV_F32 ? rhs_impl<float>(e, n, x, u, lag, dt, xdot, (cudaStream_t)stream)
                                : rhs_impl<double>(e, n, x, u, lag, dt, xdot, (cudaStream_t)stream);
}

template <typename T>
static int thruster_impl(brov_engine* e, long long n, const void* u, void* lag, double dt, void* tau, cudaStream_t st) {
    ThrusterArgs<T> a;
    int rc = make_consts<T>(e, dt, 1, &a.c);
    if (rc) return rc;
    a.u = (const T*)u; a.lag = (T*)lag; a.tau = (T*)tau; a.n = (int)n;
    CUDA_TRY(launch_thruster_wrench<T>(a, st));
    return BROV_OK;
}

extern "C" int brov_thruster_wrench(brov_engine_t* e, long long n, const void* u, void* lag, double dt, void* tau, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (e->model != BROV_THRUSTER8_LAG3) return fail(BROV_EUNSUPPORTED, "brov_thruster_wrench needs a BROV_THRUSTER8_LAG3 engine");
    if (n < 0 || n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", n);
    if (n == 0) return BROV_OK;
    if (!u || !tau) return fail(BROV_EINVAL, "u and tau must not be NULL");
    if (!(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0");
    CUDA_TRY(cudaSetDevice(e->device));
    return e->dtype == BROV_F32 ? thruster_impl<float>(e, n, u, lag, dt, tau, (cudaStream_t)stream)
                                : thruster_impl<double>(e, n, u, lag, dt, tau, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------------------
// host-buffer single calls: what `rov.dynamics(x, u, dt)` / `rov.compute_thruster_forces(u, dt)` of the model mirrors
// cost per call is launch latency, so everything travels in ONE pinned staging buffer: [in | out] -> one copy each way
// ---------------------------------------------------------------------------------------------------------------
static int call_staging(brov_engine* e, size_t bytes) {
    if (!e->call_stream) CUDA_TRY(cudaStreamCreateWithFlags(&e->call_stream, cudaStreamNonBlocking));
    if (bytes <= e->cap_call) return BROV_OK;
    size_t cap = e->cap_call ? e->cap_call : 4096;
    while (cap < bytes) cap *= 2;
    if (e->call_pinned) cudaFreeHost(e->call_pinned);
    if (e->call_dev) cudaFree(e->call_dev);
    e->call_pinned = nullptr; e->call_dev = nullptr; e->cap_call = 0;
    CUDA_TRY(cudaHostAlloc(&e->call_pinned, cap, cudaHostAllocDefault));
    CUDA_TRY(cudaMalloc(&e->call_dev, cap));
    e->cap_call = cap;
    return BROV_OK;
}

extern "C" int brov_rhs_host(brov_engine_t* e, long long n, const void* x_host, const void* u_host, void* lag_inout_host,
                             double dt, void* xdot_host) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (n < 0 || n > (1 << 24)) return fail(BROV_EINVAL, "n = %lld out of range for a host-buffer call", n);
    if (n == 0) return BROV_OK;
    if (!x_host || !u_host || !xdot_host) return fail(BROV_EINVAL, "x, u and xdot must not be NULL");
    if (e->model == BROV_THRUSTER8_LAG3 && !(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0 (it fixes the lag discretisation)");
    if (e->pv && e->pv_n != n) return fail(BROV_EINVAL, "vehicle table has %lld rows, call has n = %lld", e->pv_n, n);
    CUDA_TRY(cudaSetDevice(e->device));
    const size_t sz = scalar_size(e->dtype);
    const int NX = model_nx(e->model), NU = model_nu(e->model);
    const int NL = (e->model == BROV_THRUSTER8_LAG3 && lag_inout_host) ? 24 : 0;
    const int NXD = NX + (e->use_lag1 ? 6 : 0);
    const size_t bx = (size_t)n * NX * sz, bu = (size_t)n * NU * sz, bl = (size_t)n * NL * sz, bo = (size_t)n * NXD * sz;
    // layout: [lag | x | u | xdot]; host->device copies [lag | x | u], device->host copies back [lag] and [xdot]
    int rc = call_staging(e, bl + bx + bu + bo);
    if (rc) return rc;
    char* hp = (char*)e->call_pinned;
    char* dp = (char*)e->call_dev;
    if (NL) memcpy(hp, lag_inout_host, bl);
    memcpy(hp + bl, x_host, bx);
    memcpy(hp + bl + bx, u_host, bu);
    cudaStream_t st = e->call_stream;
    CUDA_TRY(cudaMemcpyAsync(dp, hp, bl + bx + bu, cudaMemcpyHostToDevice, st));
    rc = e->dtype == BROV_F32 ? rhs_impl<float>(e, n, dp + bl, dp + bl + bx, NL ? dp : nullptr, dt, dp + bl + bx + bu, st)
                              : rhs_impl<double>(e, n, dp + bl, dp + bl + bx, NL ? dp : nullptr, dt, dp + bl + bx + bu, st);
    if (rc) return rc;
    if (NL) CUDA_TRY(cudaMemcpyAsync(hp, dp, bl, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(hp + bl + bx + bu, dp + bl + bx + bu, bo, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (NL) memcpy(lag_inout_host, hp, bl);
    memcpy(xdot_host, hp + bl + bx + bu, bo);
    return BROV_OK;
}

extern "C" int brov_thruster_wrench_host(brov_engine_t* e, long long n, const void* u_host, void* lag_inout_host, double dt,
                                         void* tau_host) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (e->model != BROV_THRUSTER8_LAG3) return fail(BROV_EUNSUPPORTED, "brov_thruster_wrench_host needs a BROV_THRUSTER8_LAG3 engine");
    if (n < 0 || n > (1 << 24)) return fail(BROV_EINVAL, "n = %lld out of range for a host-buffer call", n);
    if (n == 0) return BROV_OK;
    if (!u_host || !tau_host) return fail(BROV_EINVAL, "u and tau must not be NULL");
    if (!(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0");
    CUDA_TRY(cudaSetDevice(e->device));
    const size_t sz = scalar_size(e->dtype);
    const size_t bl = lag_inout_host ? (size_t)n * 24 * sz : 0, bu = (size_t)n * 8 * sz, bo = (size_t)n * 6 * sz;
    int rc = call_staging(e, bl + bu + bo);
    if (rc) return rc;
    char* hp = (char*)e->call_pinned;
    char* dp = (char*)e->call_dev;
    if (bl) memcpy(hp, lag_inout_host, bl);
    memcpy(hp + bl, u_host, bu);
    cudaStream_t st = e->call_stream;
    CUDA_TRY(cudaMemcpyAsync(dp, hp, bl + bu, cudaMemcpyHostToDevice, st));
    rc = e->dtype == BROV_F32 ? thruster_impl<float>(e, n, dp + bl, bl ? dp : nullptr, dt, dp + bl + bu, st)
                              : thruster_impl<double>(e, n, dp + bl, bl ? dp : nullptr, dt, dp + bl + bu, st);
    if (rc) return rc;
    if (bl) CUDA_TRY(cudaMemcpyAsync(hp, dp, bl, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(hp + bl + bu, dp + bl + bu, bo, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (bl) memcpy(lag_inout_host, hp, bl);
    memcpy(tau_host, hp + bl + bu, bo);
    return BROV_OK;
}

static int grow(void** p, size_t* cap, size_t need) {
    if (need <= *cap) return BROV_OK;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    cudaError_t er = cudaMalloc(p, need);
    if (er != cudaSuccess) return fail(BROV_ENOMEM, "cudaMalloc(%zu): %s", need, cudaGetErrorString(er));
    *cap = need;
    return BROV_OK;
}
enum { SCR_LAG = 0, SCR_GEN = 1, SCR_MINCOS = 2, SCR_GENSNAP = 3 };
static int scratch(brov_engine* e, int which, size_t bytes, void** out) {
    int rc = grow(&e->d_scratch[which], &e->cap_scratch[which], bytes);
    *out = e->d_scratch[which];
    return rc;
}

static int carry_depth(brov_engine* e, double dt, int nsub, long long* out);

template <typename T>
static int fill_gen(const brov_input_gen& g, int nu, InputGen<T>* out) {
    memset(out, 0, sizeof(*out));
    if (!g.enable) return BROV_OK;
    if (!(g.rho >= 0.0 && g.rho <= 1.0) || !(g.sigma >= 0.0) || !(g.clip > 0.0) || !std::isfinite(g.sigma))
        return fail(BROV_EINVAL, "input generator: need 0 <= rho <= 1, sigma >= 0, clip > 0");
    if (g.vehicle0 < 0) return fail(BROV_EINVAL, "input generator: vehicle0 < 0");
    out->on = 1;
    out->rho = (float)g.rho;
    for (int j = 0; j < 8; ++j) {
        const double sc = j < nu ? g.scale[j] : 0.0;
        if (!(sc >= 0.0) || !std::isfinite(sc)) return fail(BROV_EINVAL, "input generator: scale[%d] must be finite and >= 0", j);
        out->sigma[j] = (float)(g.sigma * sc);
        out->clip[j] = (float)(std::isfinite(g.clip) ? g.clip * sc : g.clip);
    }
    out->vehicle0 = (unsigned long long)g.vehicle0;
    out->k0 = (uint32_t)(g.seed & 0xffffffffu);
    out->k1 = (uint32_t)(g.seed >> 32);
    out->state_in = (const T*)g.state_in_dev;
    out->state_out = (T*)g.state_out_dev;
    return BROV_OK;
}

// Per-thruster lag epilogue of a rollout call (thruster model): out = state of the eight ThrusterLag filters after the
// call; in = their state before it (NULL = zeros; only consulted by calls of at most `depth` steps).
struct Lag24 {
    const void* in;
    void* out;
    bool partial;   // the caller chains several calls over the filter's memory itself (brov_rollout_host): starting a
                    // short call from zeros is intended
};

template <typename T>
static int rollout_impl(brov_engine* e, const brov_rollout_desc* d, cudaStream_t st, Lag24 l24) {
    const int NX = model_nx(e->model), NU = model_nu(e->model);
    const bool thr = e->model == BROV_THRUSTER8_LAG3;
    const int nsub = d->integrator == BROV_RK4 ? 4 : 1;
    RolloutArgs<T> a;
    memset(&a, 0, sizeof(a));
    int rc = make_consts<T>(e, d->dt, nsub, &a.c);
    if (rc) return rc;
    if ((rc = fill_gen<T>(d->gen, NU, &a.gen))) return rc;
    const bool gen = a.gen.on != 0;
    a.x0 = (const T*)d->x0_dev; a.xT = (T*)d->xT_dev; a.U = (const T*)d->u_dev;
    a.u_stride_t = d->u_stride_t; a.u_stride_n = d->u_stride_n;
    a.pv = (const T*)e->pv;
    a.traj = (T*)d->traj_dev;
    a.snap_base = d->snap_base; a.step0 = d->step0;
    a.n = (int)d->n; a.steps = (int)d->steps; a.stride = (int)(d->traj_dev ? d->stride : 1);
    const size_t ualign = (sizeof(T) == 4 && NU == 6) ? 8 : 16;
    a.u_vec = !gen && aligned(d->u_dev, ualign) && (d->u_stride_t * sizeof(T)) % ualign == 0 && (d->u_stride_n * sizeof(T)) % ualign == 0;
    a.traj_vec = d->traj_dev && aligned(d->traj_dev, 16) && ((size_t)d->n * NX * sizeof(T)) % 16 == 0;

    // lag state.  The thruster model integrates the allocation-projected filters; per-thruster states for the caller
    // come from the epilogue below.
    const bool has_lag = thr || e->use_lag1;
    const int nl_kernel = thr ? 18 : 6;
    const bool want_thr_out = thr && l24.out != nullptr;
    a.lag_in = has_lag ? (const T*)d->lag_in_dev : nullptr;
    a.lag_in_w = (thr && d->lag_in_repr == BROV_LAG_PROJECTED) ? 1 : 0;
    a.lag_out = has_lag ? (thr ? (d->lag_out_repr == BROV_LAG_PROJECTED ? (T*)d->lag_out_dev : nullptr) : (T*)d->lag_out_dev) : nullptr;
    long long depth = 0;
    if (want_thr_out) {
        if ((rc = carry_depth(e, d->dt, nsub, &depth))) return rc;
        if (d->lag_in_dev && d->lag_in_repr == BROV_LAG_PROJECTED && !l24.in && !l24.partial && d->steps < depth)
            return fail(BROV_EINVAL, "per-thruster lag states cannot be recovered from an allocation-projected lag_in in a call of fewer than %lld steps", depth);
    }

    // health accounting
    a.health.counters = (unsigned long long*)d->health_dev;
    a.health.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a.mincos = (T*)d->min_abs_cos_dev;
    a.mincos_init = d->min_abs_cos_accumulate ? 0 : 1;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));

    // Temporal tiling: when the vehicle blocks do not fill a whole number of waves of resident slots, cut the launch
    // into time slices so that ceil(blocks*Q/slots) rounds of steps/Q replace ceil(blocks/slots) rounds of steps.
    a.nvblocks = (a.n + ROLLOUT_BLOCK - 1) / ROLLOUT_BLOCK;
    a.quanta = 1; a.ticket = nullptr; a.progress = nullptr;
    const bool can_slice = a.steps >= 16;
    int Q = d->time_slices;
    if (Q == 0 && can_slice) {
        const int per_sm = rollout_blocks_per_sm<T>(e->model, d->integrator, e->use_lag1 != 0, e->pv != nullptr, gen, d->traj_dev != nullptr,
                                                     a.c.has_current != 0 || !(a.u_vec && d->u_stride_n != 0));
        const long long slots = (long long)per_sm * e->num_sms;
        Q = 1;
        if (slots > 0 && a.nvblocks > slots) {
            // Work items are handed out slice-major by a ticket, so only the LAST slice pays for the partial round:
            // (ceil(r) - r) * steps / Q block-steps per slot with r = blocks / slots; every item costs a hand-over
            // (state through L2, flag wait, block start) worth about 3 block-steps.  Measured on B200
            // (profiles/f64_launch_shape.py, 512 blocks on 296 slots): 100 steps 0.515 / 0.463 / 0.482 / 0.528 ms and
            // 400 steps 1.997 / 1.745 / 1.737 / 1.774 ms for Q = 1 / 2 / 4 / 8 — the minima of this model.
            const double r = (double)a.nvblocks / (double)slots;
            const double frac = std::ceil(r) - r;
            double best = frac * a.steps + 3.0 * r;
            for (int q = 2; q <= 8 && a.steps / q >= 8; ++q) {
                const double cost = frac * a.steps / q + 3.0 * q * r;
                if (cost < best) { best = cost; Q = q; }
            }
        }
    }
    if (Q > 1 && can_slice) {
        if (Q > a.steps) Q = a.steps;
        const size_t need = 1 + (size_t)a.nvblocks;
        if (need > e->cap_sched) {
            if (e->d_sched) cudaFree(e->d_sched);
            e->d_sched = nullptr; e->cap_sched = 0;
            cudaError_t er = cudaMalloc(&e->d_sched, need * sizeof(int));
            if (er != cudaSuccess) return fail(BROV_ENOMEM, "cudaMalloc(%zu): %s", need * sizeof(int), cudaGetErrorString(er));
            e->cap_sched = need;
        }
        CUDA_TRY(cudaMemsetAsync(e->d_sched, 0, need * sizeof(int), st));
        a.quanta = Q; a.ticket = e->d_sched; a.progress = e->d_sched + 1;
        // slices hand their state over through xT and the lag / generator / min-cos arrays: scratch where the caller
        // gave none
        void* p = nullptr;
        if (has_lag && !a.lag_out) { if ((rc = scratch(e, SCR_LAG, (size_t)a.n * nl_kernel * sizeof(T), &p))) return rc; a.lag_out = (T*)p; }
        if (gen && !a.gen.state_out) { if ((rc = scratch(e, SCR_GEN, (size_t)a.n * NU * sizeof(T), &p))) return rc; a.gen.state_out = (T*)p; }
    }
    if (a.health.counters && !a.mincos && a.quanta > 1) {
        void* p = nullptr;
        if ((rc = scratch(e, SCR_MINCOS, (size_t)a.n * sizeof(T), &p))) return rc;
        a.mincos = (T*)p; a.mincos_init = 1;
    }
    // generated inputs + per-thruster lag_out: the epilogue restarts the generator from the AR(1) state before its
    // first replayed step, which the rollout kernel snapshots on the way
    const long long tail_first = want_thr_out ? (d->steps > depth ? d->steps - depth : 0) : 0;
    if (want_thr_out && gen && tail_first > 0) {
        void* p = nullptr;
        if ((rc = scratch(e, SCR_GENSNAP, (size_t)a.n * NU * sizeof(T), &p))) return rc;
        a.gen_snap = (T*)p; a.gen_snap_step = (int)tail_first;
    }
    CUDA_TRY(launch_rollout<T>(e->model, d->integrator, e->use_lag1 != 0, a, st));

    if (want_thr_out) {
        LagTailArgs<T> t;
        memset(&t, 0, sizeof(t));
        t.c = a.c;
        t.gen = a.gen;
        t.U = a.U; t.u_stride_t = a.u_stride_t; t.u_stride_n = a.u_stride_n;
        // a call of at most `depth` steps continues from the caller's per-thruster state; a longer one has forgotten it
        t.lag_in = tail_first == 0 ? (const T*)l24.in : nullptr;
        t.lag_out = (T*)l24.out;
        t.gen_state = tail_first > 0 ? a.gen_snap : (const T*)d->gen.state_in_dev;
        t.step0 = d->step0;
        t.n = a.n; t.first = (int)tail_first; t.steps = a.steps;
        CUDA_TRY(launch_lag_tail<T>(t, st));
    }
    return BROV_OK;
}

static int check_rollout_common(brov_engine* e, int integrator, long long n, long long steps, double dt) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (integrator != BROV_RK4 && integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", integrator);
    if (n < 0 || n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", n);
    if (steps < 0 || steps > (1LL << 30)) return fail(BROV_EINVAL, "steps = %lld: at most 2^30 steps per call; continue from xT / lag_out with step0", steps);
    if (!(dt > 0.0) || !std::isfinite(dt)) return fail(BROV_EINVAL, "dt must be a positive finite number");
    if (e->pv && e->pv_n != n) return fail(BROV_EINVAL, "vehicle table has %lld rows, call has n = %lld", e->pv_n, n);
    return BROV_OK;
}

// public semantics of lag_in / lag_out -> the kernel call plus the per-thruster epilogue
static int rollout_dev(brov_engine* e, const brov_rollout_desc* d, cudaStream_t st) {
    Lag24 l24 = {nullptr, nullptr, false};
    if (e->model == BROV_THRUSTER8_LAG3) {
        if (d->lag_out_dev && d->lag_out_repr == BROV_LAG_THRUSTER) l24.out = d->lag_out_dev;
        if (d->lag_in_dev && d->lag_in_repr == BROV_LAG_THRUSTER) l24.in = d->lag_in_dev;
    }
    return e->dtype == BROV_F32 ? rollout_impl<float>(e, d, st, l24) : rollout_impl<double>(e, d, st, l24);
}

extern "C" int brov_rollout(brov_engine_t* e, const brov_rollout_desc* d, void* stream) {
    if (!d || d->struct_size != sizeof(brov_rollout_desc)) return fail(BROV_EINVAL, "brov_rollout_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    int rc = check_rollout_common(e, d->integrator, d->n, d->steps, d->dt);
    if (rc) return rc;
    if (d->n == 0) return BROV_OK;
    if (!d->x0_dev || !d->xT_dev) return fail(BROV_EINVAL, "x0 and xT must not be NULL");
    if (d->steps > 0 && !d->u_dev && !d->gen.enable) return fail(BROV_EINVAL, "u is NULL");
    if (d->u_stride_t < 0 || d->u_stride_n < 0) return fail(BROV_EINVAL, "negative input stride");
    if (d->traj_dev && d->stride < 1) return fail(BROV_EINVAL, "stride must be >= 1 with a trajectory buffer");
    if (d->time_slices < 0 || d->time_slices > 64) return fail(BROV_EINVAL, "time_slices must be 0 (auto) .. 64");
    if (d->lag_in_repr < 0 || d->lag_in_repr > 1 || d->lag_out_repr < 0 || d->lag_out_repr > 1) return fail(BROV_EINVAL, "unknown lag representation");
    if (d->step0 < 0) return fail(BROV_EINVAL, "step0 < 0");
    if (d->traj_dev && d->step0 / d->stride < d->snap_base) return fail(BROV_EINVAL, "snap_base lies after the first snapshot of this call");
    const bool thr = e->model == BROV_THRUSTER8_LAG3;
    if (thr && d->lag_in_dev && d->lag_out_dev && d->lag_in_dev == d->lag_out_dev && d->lag_in_repr != d->lag_out_repr)
        return fail(BROV_EINVAL, "lag_in and lag_out alias but differ in representation");
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->steps == 0) {
        const size_t sz = scalar_size(e->dtype);
        if (d->xT_dev != d->x0_dev)
            CUDA_TRY(cudaMemcpyAsync(d->xT_dev, d->x0_dev, (size_t)d->n * model_nx(e->model) * sz, cudaMemcpyDeviceToDevice, st));
        if (d->lag_out_dev && model_nlag(e)) {
            if (d->lag_in_dev && d->lag_in_repr != d->lag_out_repr && thr)
                return fail(BROV_EUNSUPPORTED, "a zero-step rollout cannot change the lag representation");
            const int nl = (thr && d->lag_out_repr == BROV_LAG_PROJECTED) ? 18 : model_nlag(e);
            const size_t lb = (size_t)d->n * nl * sz;
            if (d->lag_in_dev) { if (d->lag_in_dev != d->lag_out_dev) CUDA_TRY(cudaMemcpyAsync(d->lag_out_dev, d->lag_in_dev, lb, cudaMemcpyDeviceToDevice, st)); }
            else CUDA_TRY(cudaMemsetAsync(d->lag_out_dev, 0, lb, st));
        }
        if (d->gen.enable && d->gen.state_out_dev) {
            const size_t gb = (size_t)d->n * model_nu(e->model) * sz;
            if (d->gen.state_in_dev) { if (d->gen.state_in_dev != d->gen.state_out_dev) CUDA_TRY(cudaMemcpyAsync(d->gen.state_out_dev, d->gen.state_in_dev, gb, cudaMemcpyDeviceToDevice, st)); }
            else CUDA_TRY(cudaMemsetAsync(d->gen.state_out_dev, 0, gb, st));
        }
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
        return BROV_OK;
    }
    return rollout_dev(e, d, st);
}

template <typename T>
static int gen_inputs_impl(const brov_gen_inputs_desc* d, cudaStream_t st) {
    GenInputsArgs<T> a;
    memset(&a, 0, sizeof(a));
    int rc = fill_gen<T>(d->gen, d->nu, &a.gen);
    if (rc) return rc;
    a.out = (T*)d->out_dev;
    a.first = d->first; a.vstride = d->vstride; a.n_sel = d->n_sel;
    a.step0 = d->step0; a.steps = (int)d->steps;
    CUDA_TRY(launch_gen_inputs<T>(d->nu, a, st));
    return BROV_OK;
}

extern "C" int brov_generate_inputs(const brov_gen_inputs_desc* d, void* stream) {
    if (!d || d->struct_size != sizeof(brov_gen_inputs_desc)) return fail(BROV_EINVAL, "brov_gen_inputs_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (d->dtype != BROV_F64 && d->dtype != BROV_F32) return fail(BROV_EINVAL, "unknown dtype %d", d->dtype);
    if (d->nu != 8 && d->nu != 6) return fail(BROV_EINVAL, "nu must be 8 or 6");
    if (!d->gen.enable) return fail(BROV_EINVAL, "gen.enable is 0");
    if (d->first < 0 || d->vstride < 1 || d->n_sel < 0 || d->n_sel > 0x7fffffffLL) return fail(BROV_EINVAL, "vehicle selection out of range");
    if (d->step0 < 0 || d->steps < 0 || d->steps > 0x7fffffffLL) return fail(BROV_EINVAL, "step range out of range");
    if (d->n_sel == 0 || d->steps == 0) return BROV_OK;
    if (!d->out_dev) return fail(BROV_EINVAL, "out is NULL");
    CUDA_TRY(cudaSetDevice(d->device));
    return d->dtype == BROV_F32 ? gen_inputs_impl<float>(d, (cudaStream_t)stream) : gen_inputs_impl<double>(d, (cudaStream_t)stream);
}

// Replay depth of the carried lag: smallest m with ||A^m||_inf * (1 + ||b||) below 1e-22 (A, b: lag map of ONE
// integrator step, i.e. Ad^nsub and S_nsub Bd).  Thrust magnitudes are O(10^2), states O(1): far below 1 ulp.
static int carry_depth(brov_engine* e, double dt, int nsub, long long* out) {
    const LagDisc* d = lag_for_dt(e, dt);
    if (!d) return BROV_EINVAL;
    typedef long double ld;
    ld A[3][3], P[3][3], tmp[3][3];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { A[i][j] = (i == j); }
    for (int s = 0; s < nsub; ++s) {
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { ld v = 0; for (int q = 0; q < 3; ++q) v += A[i][q] * (ld)d->Ad[3 * q + j]; tmp[i][j] = v; }
        memcpy(A, tmp, sizeof(A));
    }
    memcpy(P, A, sizeof(P));
    long long m = 1;
    for (; m < 100000; ++m) {
        ld nrm = 0;
        for (int i = 0; i < 3; ++i) { ld r = 0; for (int j = 0; j < 3; ++j) r += fabsl(P[i][j]); if (r > nrm) nrm = r; }
        if (nrm < 1e-22L) break;
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { ld v = 0; for (int q = 0; q < 3; ++q) v += P[i][q] * A[q][j]; tmp[i][j] = v; }
        memcpy(P, tmp, sizeof(P));
    }
    if (m >= 100000) return fail(BROV_EUNSUPPORTED, "thruster lag is not contractive at dt = %g: no finite replay depth", dt);
    *out = m;
    return BROV_OK;
}

template <typename T>
static int thruster_series_impl(brov_engine* e, long long rows, const void* u, const void* lag0, double dt, void* tau,
                                void* lag_end, cudaStream_t st) {
    ThrusterSeriesArgs<T> a;
    int rc = make_consts<T>(e, dt, 1, &a.c);
    if (rc) return rc;
    long long depth = 0;
    if ((rc = carry_depth(e, dt, 1, &depth))) return rc;
    a.U = (const T*)u; a.lag0 = (const T*)lag0; a.tau = (T*)tau; a.lag_end = (T*)lag_end;
    a.rows = rows; a.depth = (int)depth;
    CUDA_TRY(launch_thruster_series<T>(a, st));
    return BROV_OK;
}

extern "C" int brov_thruster_wrench_series(brov_engine_t* e, long long rows, const void* u_dev, const void* lag0_dev,
                                           double dt, void* tau_dev, void* lag_end_dev, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (e->model != BROV_THRUSTER8_LAG3) return fail(BROV_EUNSUPPORTED, "brov_thruster_wrench_series needs a BROV_THRUSTER8_LAG3 engine");
    if (rows < 0 || rows > 0x7fffffffLL) return fail(BROV_EINVAL, "rows = %lld out of range", rows);
    if (rows == 0) return BROV_OK;
    if (!u_dev || !tau_dev) return fail(BROV_EINVAL, "u and tau must not be NULL");
    if (!(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0");
    CUDA_TRY(cudaSetDevice(e->device));
    return e->dtype == BROV_F32 ? thruster_series_impl<float>(e, rows, u_dev, lag0_dev, dt, tau_dev, lag_end_dev, (cudaStream_t)stream)
                                : thruster_series_impl<double>(e, rows, u_dev, lag0_dev, dt, tau_dev, lag_end_dev, (cudaStream_t)stream);
}

// One integrator step for n vehicles with one input row per vehicle: the body of the reference's simulate_physics loop
// (training/train_tank_brov2_rk4.py:386-394 RK4, train_tank_brov2_full_comparison.py:462-465 Euler) as a call.
extern "C" int brov_step(brov_engine_t* e, int integrator, long long n, const void* x_dev, const void* u_dev, double dt,
                         void* x_out_dev, void* lag_inout_dev, void* stream) {
    brov_rollout_desc d;
    memset(&d, 0, sizeof(d));
    d.struct_size = sizeof(d);
    d.integrator = integrator;
    d.n = n; d.steps = 1; d.dt = dt;
    d.x0_dev = x_dev; d.xT_dev = x_out_dev; d.u_dev = u_dev;
    d.u_stride_t = 0;
    d.u_stride_n = e ? model_nu(e->model) : 0;
    d.lag_in_dev = lag_inout_dev; d.lag_out_dev = lag_inout_dev;
    d.stride = 1;
    d.lag_in_repr = d.lag_out_repr = BROV_LAG_THRUSTER;
    d.time_slices = 1;
    return brov_rollout(e, &d, stream);
}

extern "C" int brov_se_carry_steps(brov_engine_t* e, double dt, int integrator, long long* steps_out) {
    if (!e || !steps_out) return fail(BROV_EINVAL, "NULL argument");
    if (e->model != BROV_THRUSTER8_LAG3) { *steps_out = 0; return BROV_OK; }
    if (!(dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0");
    return carry_depth(e, dt, integrator == BROV_RK4 ? 4 : 1, steps_out);
}

static constexpr int SE_MAX_QUANTA = 4;
static size_t se_align(size_t b) { return (b + 255) & ~(size_t)255; }
// partial sums (per block and time slice), ticket + progress flags, and the hand-over rows of the time slices
// (state 13 + lag 18 scalars, min |cos theta|, non-finite flag per window)
static size_t se_partial_bytes(long long n_windows) {
    return se_align((size_t)((n_windows + 63) / 64) * SE_MAX_QUANTA * MAX_H * sizeof(double));  // blocks down to 64 windows
}
static size_t se_flag_bytes(long long n_windows) { return se_align((size_t)(2 + (n_windows + 63) / 64) * sizeof(int)); }
extern "C" size_t brov_se_workspace_bytes(long long n_windows) {
    if (n_windows < 1) n_windows = 1;
    return se_partial_bytes(n_windows) + se_flag_bytes(n_windows) + se_align((size_t)n_windows * 13 * sizeof(double)) +
           se_align((size_t)n_windows * 18 * sizeof(double)) + 2 * se_align((size_t)n_windows * 4);
}

// Windows per thread of a carried-lag pass: the replay (m lag-only steps, each about a fifth of a full step: 152 of 838
// FP64 operations) is paid once per wpt windows of H steps each; more windows per thread mean fewer threads — pick the
// count that minimises rounds x work per thread (any count up to 64, not only powers of two: with 1M windows of
// H = 100, wpt = 7 fills 3.77 -> 4 rounds, wpt = 4 fills 6.6 -> 7)
static int carry_wpt(const brov_engine* e, long long n_windows, long long H, long long m) {
    const double slots = 2.0 * e->num_sms * ROLLOUT_BLOCK * (e->dtype == BROV_F32 ? 2.0 : 1.0);
    double best = 1e300;
    int wpt = 1;
    for (int w = 1; w <= 64; ++w) {
        const double threads = std::ceil((double)n_windows / w);
        const double cost = std::ceil(threads / slots) * ((double)w * (double)H + 0.2 * (double)m);
        if (cost < best * 0.98) { best = cost; wpt = w; }
    }
    return wpt;
}
// the replay of window0's history reads input rows back to window (window0 * H - m) / H: they must be local
static int check_carry_rows(long long window0, long long row0, long long H, long long m) {
    const long long first_hist = window0 * H - m;
    const long long need_row = first_hist > 0 ? first_hist / H : 0;
    if (row0 > need_row)
        return fail(BROV_EINVAL, "lag_carry: the shard must start at row %lld or earlier (row0 = %lld): window %lld replays %lld steps of history", need_row, row0, window0, m);
    return BROV_OK;
}

template <typename T>
static int se_impl(brov_engine* e, const brov_se_desc* d, cudaStream_t st) {
    SeArgs<T> a;
    int rc = make_consts<T>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a.c);
    if (rc) return rc;
    a.X = (const T*)d->X_dev; a.U = (const T*)d->U_dev; a.lag0 = (const T*)d->lag0_dev;
    a.partial = (double*)d->workspace_dev;
    a.rows = (int)d->rows; a.nwin = (int)d->n_windows; a.nH = d->n_horizons;
    for (int h = 0; h < MAX_H; ++h) a.H[h] = h < d->n_horizons ? d->horizons[h] : 0x7fffffff;
    a.carry_steps = 0; a.wpt = 1; a.win0 = d->window0; a.row0 = d->row0;
    if (d->lag_carry && e->model == BROV_THRUSTER8_LAG3) {
        long long m = 0;
        if ((rc = carry_depth(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &m))) return rc;
        a.carry_steps = (int)m;
        a.wpt = carry_wpt(e, d->n_windows, d->horizons[0], m);
        if ((rc = check_carry_rows(d->window0, d->row0, d->horizons[0], m))) return rc;
    }
    a.health.counters = (unsigned long long*)d->health_dev;
    a.health.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    // Temporal tiling against wave quantisation (SeArgs::quanta): reset mode only (a carried-lag thread walks several
    // windows in sequence).  Q slices cost ceil(blocks Q / slots) / Q rounds of the longest horizon, plus ~1 % per
    // extra slice for the hand-over through memory.
    a.quanta = 1; a.nwblocks = se_blocks<T>(a.nwin); a.ticket = nullptr; a.progress = nullptr;
    a.st_x = nullptr; a.st_lag = nullptr; a.st_mc = nullptr; a.st_bad = nullptr;
    if (a.wpt == 1 && a.carry_steps == 0 && a.nwin > 0) {
        const int hmax = d->horizons[d->n_horizons - 1];
        const double slots = 2.0 * e->num_sms * (e->dtype == BROV_F32 ? 2.0 : 1.0);
        if (d->time_slices == 0) {
            double best = std::ceil(a.nwblocks / slots);
            for (int q = 2; q <= SE_MAX_QUANTA && hmax >= 8 * q; ++q) {
                const double cost = std::ceil((double)a.nwblocks * q / slots) / q * (1.0 + 0.01 * (q - 1));
                if (cost < best * 0.97) { best = cost; a.quanta = q; }
            }
        } else {
            a.quanta = d->time_slices < hmax ? d->time_slices : hmax;
        }
        if (a.quanta > 1) {
            unsigned char* w = (unsigned char*)d->workspace_dev + se_partial_bytes(d->n_windows);
            a.ticket = (int*)w; a.progress = a.ticket + 1;
            CUDA_TRY(cudaMemsetAsync(w, 0, (size_t)(1 + a.nwblocks) * sizeof(int), st));
            w += se_flag_bytes(d->n_windows);
            a.st_x = (T*)w; w += se_align((size_t)d->n_windows * 13 * sizeof(double));
            a.st_lag = (T*)w; w += se_align((size_t)d->n_windows * 18 * sizeof(double));
            a.st_mc = (float*)w; w += se_align((size_t)d->n_windows * 4);
            a.st_bad = (int*)w;
        }
    }
    CUDA_TRY(launch_se<T>(e->model, d->integrator, a, d->se_out_dev, st));
    return BROV_OK;
}

// argument checks of the sliding-window geometry shared by brov_multistep_se and brov_multistep_se_sweep
template <class D> static int check_se_geometry(const D* d) {
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (d->n_horizons < 1 || d->n_horizons > MAX_H) return fail(BROV_EINVAL, "n_horizons must be 1..%d", MAX_H);
    if (d->lag_carry && (d->n_horizons != 1 || d->lag0_dev)) return fail(BROV_EINVAL, "lag_carry scores one horizon per call and excludes lag0");
    if (d->window0 < 0 || d->row0 < 0 || d->row0 > d->window0) return fail(BROV_EINVAL, "window0 / row0 out of range");
    if (!d->lag_carry && (d->window0 != d->row0)) return fail(BROV_EINVAL, "rows before the first window are only meaningful with lag_carry");
    for (int h = 0; h < d->n_horizons; ++h)
        if (d->horizons[h] < 1 || d->horizons[h] > (1 << 29) || (h && d->horizons[h] <= d->horizons[h - 1])) return fail(BROV_EINVAL, "horizons must be in [1, 2^29] and strictly ascending");
    if (d->rows < 0 || d->rows > 0x7fffffffLL || d->n_windows < 0 || d->n_windows > d->rows) return fail(BROV_EINVAL, "rows / n_windows out of range");
    // every window's first row must be local: window k starts at local row k + (window0 - row0)
    if (d->n_windows + (d->window0 - d->row0) > d->rows)
        return fail(BROV_EINVAL, "n_windows = %lld starting at local row %lld exceed the %lld rows of the series", d->n_windows, d->window0 - d->row0, d->rows);
    if (!(d->dt > 0.0)) return fail(BROV_EINVAL, "dt must be > 0");
    return BROV_OK;
}
// count_out (host, may be NULL): the number of windows that reach each horizon
template <class D> static void se_counts(const D* d) {
    for (int h = 0; h < MAX_H; ++h) {
        long long cnt = 0;
        if (h < d->n_horizons) {
            cnt = d->rows - (d->window0 - d->row0) - d->horizons[h];
            if (cnt > d->n_windows) cnt = d->n_windows;
            if (cnt < 0) cnt = 0;
        }
        if (d->count_out) d->count_out[h] = cnt;
    }
}

extern "C" int brov_multistep_se(brov_engine_t* e, const brov_se_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_se_desc)) return fail(BROV_EINVAL, "brov_se_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "the evaluator does not support the first-order wrench lag");
    if (e->pv) return fail(BROV_EUNSUPPORTED, "the evaluator scores one vehicle; clear the per-vehicle table first");
    int rc = check_se_geometry(d);
    if (rc) return rc;
    if (!d->se_out_dev) return fail(BROV_EINVAL, "se_out is NULL");
    CUDA_TRY(cudaSetDevice(e->device));
    se_counts(d);
    if (d->n_windows == 0 || d->rows < 2) {
        CUDA_TRY(cudaMemsetAsync(d->se_out_dev, 0, MAX_H * sizeof(double), (cudaStream_t)stream));
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), (cudaStream_t)stream));
        return BROV_OK;
    }
    if (!d->X_dev || !d->U_dev) return fail(BROV_EINVAL, "X and U must not be NULL");
    if (d->time_slices < 0 || d->time_slices > SE_MAX_QUANTA) return fail(BROV_EINVAL, "time_slices must be 0 (automatic) .. %d", SE_MAX_QUANTA);
    if (!d->workspace_dev || d->workspace_bytes < brov_se_workspace_bytes(d->n_windows)) return fail(BROV_EINVAL, "workspace too small: need %zu bytes", brov_se_workspace_bytes(d->n_windows));
    return e->dtype == BROV_F32 ? se_impl<float>(e, d, (cudaStream_t)stream) : se_impl<double>(e, d, (cudaStream_t)stream);
}

// sweep workspace: per-candidate partial sums [P][window blocks][MAX_H], then (carry mode) the lag each window inherits
// [n_windows][18] (sized for fp64 whatever the engine's scalar type)
static size_t sweep_partial_bytes(long long n_candidates, long long n_windows) {
    return se_align((size_t)n_candidates * (size_t)((n_windows + ROLLOUT_BLOCK - 1) / ROLLOUT_BLOCK) * MAX_H * sizeof(double));
}
extern "C" size_t brov_se_sweep_workspace_bytes(long long n_candidates, long long n_windows, int lag_carry) {
    if (n_candidates < 0) n_candidates = 0;
    if (n_windows < 0) n_windows = 0;
    return sweep_partial_bytes(n_candidates, n_windows) + (lag_carry ? se_align((size_t)n_windows * 18 * sizeof(double)) : 0);
}

template <typename T>
static int se_sweep_impl(brov_engine* e, const brov_se_sweep_desc* d, cudaStream_t st) {
    SweepArgs<T> a;
    memset(&a, 0, sizeof(a));
    const int nsub = d->integrator == BROV_RK4 ? 4 : 1;
    int rc = make_consts<T>(e, d->dt, nsub, &a.c);
    if (rc) return rc;
    a.c.has_current = d->any_current ? 1 : 0;   // the candidates' currents, not the engine's
    a.X = (const T*)d->X_dev; a.U = (const T*)d->U_dev;
    a.kp = (const T*)d->kp_soa_dev;
    a.partial = (double*)d->workspace_dev;
    a.health = (unsigned long long*)d->health_dev;
    a.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a.off = d->window0 - d->row0;
    a.rows = (int)d->rows; a.nwin = (int)d->n_windows; a.nH = d->n_horizons;
    for (int h = 0; h < MAX_H; ++h) a.H[h] = h < d->n_horizons ? d->horizons[h] : 0x7fffffff;
    a.P = (int)d->n_candidates;
    a.nwb = se_blocks<T>(a.nwin);
    a.lag0 = (const T*)d->lag0_dev;
    a.lag0_w = 0;
    if (d->lag_carry && e->model == BROV_THRUSTER8_LAG3) {
        long long m = 0;
        if ((rc = carry_depth(e, d->dt, nsub, &m))) return rc;
        if ((rc = check_carry_rows(d->window0, d->row0, d->horizons[0], m))) return rc;
        CarryLagArgs<T> c;
        memset(&c, 0, sizeof(c));
        c.c = a.c;
        c.U = a.U;
        c.lag_out = (T*)((unsigned char*)d->workspace_dev + sweep_partial_bytes(d->n_candidates, d->n_windows));
        c.win0 = d->window0; c.row0 = d->row0;
        c.rows = a.rows; c.nwin = a.nwin; c.H = d->horizons[0]; c.carry_steps = (int)m;
        c.wpt = carry_wpt(e, d->n_windows, d->horizons[0], m);
        CUDA_TRY(launch_se_carry_lag<T>(c, st));
        a.lag0 = c.lag_out;
        a.lag0_w = 1;
    }
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, (size_t)d->n_candidates * 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_se_sweep<T>(e->model, d->integrator, a, d->se_out_dev, st));
    return BROV_OK;
}

extern "C" int brov_multistep_se_sweep(brov_engine_t* e, const brov_se_sweep_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_se_sweep_desc)) return fail(BROV_EINVAL, "brov_se_sweep_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "the sweep serves the Fossen models; double-integrator engines have no coefficient table");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "the evaluator does not support the first-order wrench lag");
    int rc = check_se_geometry(d);
    if (rc) return rc;
    if (d->n_candidates < 0) return fail(BROV_EINVAL, "n_candidates = %lld", d->n_candidates);
    const long long nwb = (d->n_windows + ROLLOUT_BLOCK - 1) / ROLLOUT_BLOCK;
    if (d->n_candidates * nwb > 0x7fffffffLL)
        return fail(BROV_EINVAL, "%lld candidates x %lld window blocks exceed 2^31 - 1 blocks: split the candidates over several calls", d->n_candidates, nwb);
    se_counts(d);
    if (d->n_candidates == 0) return BROV_OK;
    if (!d->se_out_dev) return fail(BROV_EINVAL, "se_out is NULL");
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->n_windows == 0 || d->rows < 2) {
        CUDA_TRY(cudaMemsetAsync(d->se_out_dev, 0, (size_t)d->n_candidates * MAX_H * sizeof(double), st));
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, (size_t)d->n_candidates * 2 * sizeof(unsigned long long), st));
        return BROV_OK;
    }
    if (!d->X_dev || !d->U_dev) return fail(BROV_EINVAL, "X and U must not be NULL");
    if (!d->kp_soa_dev) return fail(BROV_EINVAL, "kp_soa is NULL");
    const size_t need = brov_se_sweep_workspace_bytes(d->n_candidates, d->n_windows, d->lag_carry && e->model == BROV_THRUSTER8_LAG3);
    if (!d->workspace_dev || d->workspace_bytes < need) return fail(BROV_EINVAL, "workspace too small: need %zu bytes", need);
    return e->dtype == BROV_F32 ? se_sweep_impl<float>(e, d, st) : se_sweep_impl<double>(e, d, st);
}

// gradient workspace: per-block partials [GRAD_MAX_GRID][MAX_H][1 + p + p(p+1)/2], then (carry mode) the lag each
// window inherits [n_windows][18]
static size_t grad_partial_bytes(int n_dirs) {
    const size_t ne = 1 + (size_t)n_dirs + (size_t)n_dirs * (n_dirs + 1) / 2;
    return se_align((size_t)GRAD_MAX_GRID * MAX_H * ne * sizeof(double));
}
extern "C" size_t brov_se_grad_workspace_bytes(long long n_windows, int n_dirs, int lag_carry) {
    if (n_windows < 0) n_windows = 0;
    if (n_dirs < 1 || n_dirs > KP_COUNT) return 0;
    return grad_partial_bytes(n_dirs) + (lag_carry ? se_align((size_t)n_windows * 18 * sizeof(double)) : 0);
}

static int se_grad_impl(brov_engine* e, const brov_se_grad_desc* d, cudaStream_t st) {
    GradArgs a;
    memset(&a, 0, sizeof(a));
    const int nsub = d->integrator == BROV_RK4 ? 4 : 1;
    int rc = make_consts<double>(e, d->dt, nsub, &a.c);
    if (rc) return rc;
    a.c.has_current = d->any_current ? 1 : 0;   // the point's and the directions' currents, not the engine's
    a.X = (const double*)d->X_dev; a.U = (const double*)d->U_dev;
    a.kp = d->kp_dev; a.dirs = d->dirs_dev;
    a.partial = (double*)d->workspace_dev;
    a.health = (unsigned long long*)d->health_dev;
    a.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a.off = d->window0 - d->row0;
    a.rows = (int)d->rows; a.nwin = (int)d->n_windows; a.nH = d->n_horizons;
    for (int h = 0; h < MAX_H; ++h) a.H[h] = h < d->n_horizons ? d->horizons[h] : 0x7fffffff;
    a.p = d->n_dirs;
    a.W = GRAD_BLOCK / a.p;
    a.ntiles = (int)((d->n_windows + a.W - 1) / a.W);
    a.ne = 1 + a.p + a.p * (a.p + 1) / 2;
    a.lag0 = (const double*)d->lag0_dev;
    a.lag0_w = 0;
    if (d->lag_carry && e->model == BROV_THRUSTER8_LAG3) {
        // the inherited lag does not depend on the coefficients: the sweep's pre-pass serves every direction
        long long m = 0;
        if ((rc = carry_depth(e, d->dt, nsub, &m))) return rc;
        if ((rc = check_carry_rows(d->window0, d->row0, d->horizons[0], m))) return rc;
        CarryLagArgs<double> c;
        memset(&c, 0, sizeof(c));
        c.c = a.c;
        c.U = a.U;
        c.lag_out = (double*)((unsigned char*)d->workspace_dev + grad_partial_bytes(d->n_dirs));
        c.win0 = d->window0; c.row0 = d->row0;
        c.rows = a.rows; c.nwin = a.nwin; c.H = d->horizons[0]; c.carry_steps = (int)m;
        c.wpt = carry_wpt(e, d->n_windows, d->horizons[0], m);
        CUDA_TRY(launch_se_carry_lag<double>(c, st));
        a.lag0 = c.lag_out;
        a.lag0_w = 1;
    }
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_se_grad(e->model, d->integrator, a, e->num_sms, d->se_out_dev, d->grad_out_dev, d->gn_out_dev, st));
    return BROV_OK;
}

extern "C" int brov_multistep_se_grad(brov_engine_t* e, const brov_se_grad_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_se_grad_desc)) return fail(BROV_EINVAL, "brov_se_grad_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "the gradient serves the Fossen models; double-integrator engines have no coefficient table");
    if (e->dtype != BROV_F64) return fail(BROV_EUNSUPPORTED, "the gradient is computed in fp64: create the engine with BROV_F64");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "the evaluator does not support the first-order wrench lag");
    int rc = check_se_geometry(d);
    if (rc) return rc;
    if (d->n_dirs < 1 || d->n_dirs > KP_COUNT) return fail(BROV_EINVAL, "n_dirs = %d must be 1..%d", d->n_dirs, KP_COUNT);
    if (!d->se_out_dev || !d->grad_out_dev || !d->gn_out_dev) return fail(BROV_EINVAL, "se_out, grad_out and gn_out must not be NULL");
    se_counts(d);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->n_windows == 0 || d->rows < 2) {
        const size_t p = (size_t)d->n_dirs;
        CUDA_TRY(cudaMemsetAsync(d->se_out_dev, 0, MAX_H * sizeof(double), st));
        CUDA_TRY(cudaMemsetAsync(d->grad_out_dev, 0, MAX_H * p * sizeof(double), st));
        CUDA_TRY(cudaMemsetAsync(d->gn_out_dev, 0, MAX_H * p * p * sizeof(double), st));
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
        return BROV_OK;
    }
    if (!d->X_dev || !d->U_dev) return fail(BROV_EINVAL, "X and U must not be NULL");
    if (!d->kp_dev || !d->dirs_dev) return fail(BROV_EINVAL, "kp and dirs must not be NULL");
    const size_t need = brov_se_grad_workspace_bytes(d->n_windows, d->n_dirs, d->lag_carry && e->model == BROV_THRUSTER8_LAG3);
    if (!d->workspace_dev || d->workspace_bytes < need) return fail(BROV_EINVAL, "workspace too small: need %zu bytes", need);
    return se_grad_impl(e, d, st);
}

extern "C" int brov_linearize(brov_engine_t* e, const brov_linearize_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_linearize_desc)) return fail(BROV_EINVAL, "brov_linearize_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "linearize serves the Fossen models, not double-integrator engines");
    if (e->dtype != BROV_F64) return fail(BROV_EUNSUPPORTED, "the Jacobians are computed in fp64: create the engine with BROV_F64");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "linearize does not support the first-order wrench lag");
    if (e->pv) return fail(BROV_EUNSUPPORTED, "linearize uses the shared coefficients: clear the per-vehicle table first");
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (d->n < 0 || d->n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", d->n);
    if (d->steps < 1 || d->steps > (1LL << 30)) return fail(BROV_EINVAL, "steps = %lld must be 1 .. 2^30", d->steps);
    if (!(d->dt > 0.0) || !std::isfinite(d->dt)) return fail(BROV_EINVAL, "dt must be a positive finite number");
    if (!d->jac_dev) return fail(BROV_EINVAL, "jac is NULL");
    if (!d->z0_dev || !d->u_dev) return fail(BROV_EINVAL, "z0 and u must not be NULL");
    if (d->u_stride_t < 0 || d->u_stride_n < 0) return fail(BROV_EINVAL, "negative input stride");
    if (d->n == 0) return BROV_OK;
    LinArgs a;
    memset(&a, 0, sizeof(a));
    int rc = make_consts<double>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a.c);
    if (rc) return rc;
    a.z0 = (const double*)d->z0_dev;
    a.U = (const double*)d->u_dev;
    a.ust = d->u_stride_t; a.usn = d->u_stride_n;
    a.z_out = (double*)d->z_out_dev;
    a.z_traj = (double*)d->z_traj_dev;
    a.jac = (double*)d->jac_dev;
    a.health = (unsigned long long*)d->health_dev;
    a.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a.n = d->n;
    a.steps = (int)d->steps;
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_linearize(e->model, d->integrator, a, st));
    return BROV_OK;
}

// The checks brov_closed_loop and brov_closed_loop_vjp share, in this order: integrator, n, steps (min_steps ..
// 2^30), dt, operand strides, input bounds, the stride of a trajectory buffer or cotangent (`traj`, named traj_what),
// the rows of the vehicle table and, when n > 0, the state pointers (z0 and `out`, named in out_what) and the
// operands.  A caller with nothing left to do for n = 0 returns after it.
template <class Desc>
static int cl_check(const brov_engine* e, const Desc* d, long long min_steps, bool traj, const char* traj_what,
                    const void* out, const char* out_what) {
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (d->n < 0 || d->n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", d->n);
    if (d->steps < min_steps || d->steps > (1LL << 30))
        return fail(BROV_EINVAL, "steps = %lld must be %lld .. 2^30", d->steps, min_steps);
    if (!(d->dt > 0.0) || !std::isfinite(d->dt)) return fail(BROV_EINVAL, "dt must be a positive finite number");
    if (d->K_stride_t < 0 || d->K_stride_n < 0 || d->z_ref_stride_t < 0 || d->z_ref_stride_n < 0 || d->u_ref_stride_t < 0 ||
        d->u_ref_stride_n < 0)
        return fail(BROV_EINVAL, "negative operand stride");
    for (int r = 0; r < model_nu(e->model); ++r)
        if (std::isnan(d->u_min[r]) || std::isnan(d->u_max[r]) || d->u_min[r] > d->u_max[r])
            return fail(BROV_EINVAL, "input bounds of channel %d: u_min = %g, u_max = %g", r, d->u_min[r], d->u_max[r]);
    if (traj && d->stride < 1) return fail(BROV_EINVAL, "stride must be >= 1 with a %s", traj_what);
    if (e->pv && e->pv_n != d->n) return fail(BROV_EINVAL, "vehicle table has %lld rows, call has n = %lld", e->pv_n, d->n);
    if (d->n == 0) return BROV_OK;
    if (!d->z0_dev || !out) return fail(BROV_EINVAL, "z0 and %s must not be NULL", out_what);
    if (d->steps > 0 && (!d->K_dev || !d->z_ref_dev || !d->u_ref_dev)) return fail(BROV_EINVAL, "K, z_ref and u_ref must not be NULL");
    return BROV_OK;
}

// the operand fields of ClArgs<T> / ClAdjArgs from a closed-loop descriptor: K, z_ref and u_ref with their strides,
// the shared-memory K, the vehicle table, the bounds, the cost weights (zero past nu / NZ) and eps
template <class Args, class Desc>
static void cl_operands(const brov_engine* e, const Desc* d, Args* a) {
    using T = typename std::remove_const<typename std::remove_pointer<decltype(a->K)>::type>::type;
    const int nz = model_nz(e->model), nu = model_nu(e->model);
    a->K = (const T*)d->K_dev; a->K_st = d->K_stride_t; a->K_sn = d->K_stride_n;
    a->zr = (const T*)d->z_ref_dev; a->zr_st = d->z_ref_stride_t; a->zr_sn = d->z_ref_stride_n;
    a->ur = (const T*)d->u_ref_dev; a->ur_st = d->u_ref_stride_t; a->ur_sn = d->u_ref_stride_n;
    a->k_smem = (a->K_st == 0 && a->K_sn == 0) ? 1 : 0;
    a->pv = (const T*)e->pv;
    a->eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    for (int r = 0; r < 8; ++r) { a->u_min[r] = (T)d->u_min[r]; a->u_max[r] = (T)d->u_max[r]; a->r[r] = r < nu ? (T)d->r[r] : T(0); }
    for (int j = 0; j < CL_MAX_NZ; ++j) a->q[j] = j < nz ? (T)d->q[j] : T(0);
}

template <typename T>
static int closed_loop_impl(brov_engine* e, const brov_closed_loop_desc* d, int nz, int nu, cudaStream_t st) {
    ClArgs<T> a;
    memset(&a, 0, sizeof(a));
    int rc = make_consts<T>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a.c);
    if (rc) return rc;
    cl_operands(e, d, &a);
    a.z0 = (const T*)d->z0_dev;
    a.z_out = (T*)d->z_out_dev;
    a.traj = (T*)d->traj_dev;
    a.u_traj = (T*)d->u_traj_dev;
    a.cost = (T*)d->cost_dev;
    a.cost_accumulate = d->cost_accumulate ? 1 : 0;
    a.health = (unsigned long long*)d->health_dev;
    a.n = d->n;
    a.steps = (int)d->steps;
    a.stride = (d->traj_dev || d->u_traj_dev) ? (int)std::min<long long>(d->stride, 0x7fffffffLL) : 0x7fffffff;
    a.traj_vec = d->traj_dev && aligned(d->traj_dev, 16) && ((size_t)d->n * nz * sizeof(T)) % 16 == 0;
    a.u_traj_vec = d->u_traj_dev && aligned(d->u_traj_dev, 16) && ((size_t)d->n * nu * sizeof(T)) % 16 == 0;
    // Threads per block: 128 once that still gives every SM a block, else 64 or 32 — one thread per vehicle leaves
    // most SMs idle at small n (4096 vehicles in 128-thread blocks occupy 32 of 148 SMs)
    int block = 128;
    while (block > 32 && (d->n + block - 1) / block < e->num_sms) block /= 2;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_closed_loop<T>(e->model, d->integrator, block, a, st));
    return BROV_OK;
}

extern "C" int brov_closed_loop(brov_engine_t* e, const brov_closed_loop_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_closed_loop_desc)) return fail(BROV_EINVAL, "brov_closed_loop_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "closed_loop serves the Fossen models, not double-integrator engines");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "closed_loop does not support the first-order wrench lag");
    int rc = cl_check(e, d, 0, d->traj_dev || d->u_traj_dev, "trajectory buffer", d->z_out_dev, "z_out");
    if (rc || d->n == 0) return rc;
    const int nz = model_nz(e->model), nu = model_nu(e->model);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->steps == 0) {
        const size_t sz = scalar_size(e->dtype);
        if (d->z_out_dev != d->z0_dev)
            CUDA_TRY(cudaMemcpyAsync(d->z_out_dev, d->z0_dev, (size_t)d->n * nz * sz, cudaMemcpyDeviceToDevice, st));
        if (d->cost_dev && !d->cost_accumulate) CUDA_TRY(cudaMemsetAsync(d->cost_dev, 0, (size_t)d->n * sz, st));
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
        return BROV_OK;
    }
    return e->dtype == BROV_F32 ? closed_loop_impl<float>(e, d, nz, nu, st) : closed_loop_impl<double>(e, d, nz, nu, st);
}

// the noise variances are read back and checked on the host before the launch: q >= 0, r > 0 (a NaN fails both)
static int check_noise(const void* dev, long long sn, long long n, int nx, bool strict, const char* what, cudaStream_t st) {
    const size_t cnt = (size_t)(sn ? (n - 1) * sn + nx : nx);
    std::vector<double> h(cnt);
    CUDA_TRY(cudaMemcpyAsync(h.data(), dev, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (long long i = 0; i < (sn ? n : 1); ++i)
        for (int j = 0; j < nx; ++j) {
            const double v = h[(size_t)(i * sn + j)];
            if (!(strict ? v > 0.0 : v >= 0.0) || !std::isfinite(v))
                return fail(BROV_EINVAL, "%s[%lld][%d] = %g must be %s", what, sn ? i : 0LL, j, v,
                            strict ? "positive and finite" : "non-negative and finite");
        }
    return BROV_OK;
}

extern "C" int brov_ekf(brov_engine_t* e, const brov_ekf_desc* d, void* stream) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (!d || d->struct_size != sizeof(brov_ekf_desc)) return fail(BROV_EINVAL, "brov_ekf_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "ekf serves the Fossen models, not double-integrator engines");
    if (e->model == BROV_WRENCH_QUAT13)
        return fail(BROV_EUNSUPPORTED, "ekf does not serve quat13: the covariance of a unit quaternion is singular (use wrench12)");
    if (e->dtype != BROV_F64) return fail(BROV_EUNSUPPORTED, "the filter runs in fp64: create the engine with BROV_F64");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "ekf does not support the first-order wrench lag");
    if (e->pv) return fail(BROV_EUNSUPPORTED, "ekf uses the shared coefficients: clear the per-vehicle table first");
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (d->n < 0 || d->n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", d->n);
    if (d->steps < 0 || d->steps > (1LL << 30)) return fail(BROV_EINVAL, "steps = %lld must be 0 .. 2^30", d->steps);
    if (!(d->dt > 0.0) || !std::isfinite(d->dt)) return fail(BROV_EINVAL, "dt must be a positive finite number");
    if (d->u_stride_t < 0 || d->u_stride_n < 0 || d->y_stride_t < 0 || d->y_stride_n < 0 || d->q_stride_n < 0 ||
        d->r_stride_n < 0)
        return fail(BROV_EINVAL, "negative operand stride");
    if ((d->x_traj_dev || d->P_traj_dev) && d->stride < 1) return fail(BROV_EINVAL, "stride must be >= 1 with a trajectory buffer");
    const bool stats = d->loglik_dev || d->nis_dev || d->count_dev;
    if (stats && !(d->loglik_dev && d->nis_dev && d->count_dev)) return fail(BROV_EINVAL, "loglik, nis and count go together");
    if (d->n == 0) return BROV_OK;
    if (!d->z0_dev || !d->P0_dev || !d->z_out_dev || !d->P_out_dev) return fail(BROV_EINVAL, "z0, P0, z_out and P_out must not be NULL");
    const int nx = model_nx(e->model), nz = model_nz(e->model);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->steps == 0) {
        if (d->z_out_dev != d->z0_dev)
            CUDA_TRY(cudaMemcpyAsync(d->z_out_dev, d->z0_dev, (size_t)d->n * nz * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (d->P_out_dev != d->P0_dev)
            CUDA_TRY(cudaMemcpyAsync(d->P_out_dev, d->P0_dev, (size_t)d->n * nx * nx * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (stats && !d->stats_accumulate) {
            CUDA_TRY(cudaMemsetAsync(d->loglik_dev, 0, (size_t)d->n * sizeof(double), st));
            CUDA_TRY(cudaMemsetAsync(d->nis_dev, 0, (size_t)d->n * sizeof(double), st));
            CUDA_TRY(cudaMemsetAsync(d->count_dev, 0, (size_t)d->n * sizeof(long long), st));
        }
        if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
        return BROV_OK;
    }
    if (!d->u_dev || !d->y_dev || !d->q_dev || !d->r_dev) return fail(BROV_EINVAL, "u, y, q and r must not be NULL");
    int rc = check_noise(d->q_dev, d->q_stride_n, d->n, nx, false, "q", st);
    if (rc) return rc;
    if ((rc = check_noise(d->r_dev, d->r_stride_n, d->n, nx, true, "r", st))) return rc;
    EkfArgs a;
    memset(&a, 0, sizeof(a));
    if ((rc = make_consts<double>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a.c))) return rc;
    a.z0 = (const double*)d->z0_dev;
    a.P0 = (const double*)d->P0_dev;
    a.U = (const double*)d->u_dev; a.ust = d->u_stride_t; a.usn = d->u_stride_n;
    a.Y = (const double*)d->y_dev; a.yst = d->y_stride_t; a.ysn = d->y_stride_n;
    a.q = (const double*)d->q_dev; a.qsn = d->q_stride_n;
    a.r = (const double*)d->r_dev; a.rsn = d->r_stride_n;
    a.z_out = (double*)d->z_out_dev;
    a.P_out = (double*)d->P_out_dev;
    a.x_traj = (double*)d->x_traj_dev;
    a.P_traj = (double*)d->P_traj_dev;
    a.loglik = (double*)d->loglik_dev;
    a.nis = (double*)d->nis_dev;
    a.count = (long long*)d->count_dev;
    a.accumulate = d->stats_accumulate ? 1 : 0;
    a.health = (unsigned long long*)d->health_dev;
    a.eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a.n = d->n;
    a.steps = (int)d->steps;
    a.stride = (d->x_traj_dev || d->P_traj_dev) ? (int)std::min<long long>(d->stride, 0x7fffffffLL) : 0x7fffffff;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_ekf(e->model, d->integrator, a, st));
    return BROV_OK;
}

extern "C" size_t brov_rollout_vjp_workspace_bytes(int model, long long n, long long steps) {
    if (model != BROV_THRUSTER8_LAG3 && model != BROV_WRENCH_EULER12 && model != BROV_WRENCH_QUAT13) return 0;
    return adjoint_workspace_bytes(model_nz(model), n, steps);
}

// the argument checks of brov_rollout_vjp / brov_rollout_vjp_coef in order, then (n > 0) the kernel arguments a and the
// health counters zeroed on st
static int rollout_vjp_args(brov_engine_t* e, const brov_rollout_vjp_desc* d, AdjArgs* a, cudaStream_t st) {
    if (d->integrator != BROV_RK4 && d->integrator != BROV_EULER) return fail(BROV_EINVAL, "unknown integrator %d", d->integrator);
    if (d->n < 0 || d->n > 0x7fffffffLL) return fail(BROV_EINVAL, "n = %lld out of range", d->n);
    if (d->steps < 1 || d->steps > (1LL << 30)) return fail(BROV_EINVAL, "steps = %lld must be 1 .. 2^30", d->steps);
    if (!(d->dt > 0.0) || !std::isfinite(d->dt)) return fail(BROV_EINVAL, "dt must be a positive finite number");
    if (d->u_stride_t < 0 || d->u_stride_n < 0) return fail(BROV_EINVAL, "negative input stride");
    if (d->gtraj_dev && d->stride < 1) return fail(BROV_EINVAL, "stride must be >= 1 with a trajectory cotangent");
    if (d->n == 0) return BROV_OK;
    if (!d->z0_dev || !d->u_dev || !d->gz0_dev || !d->gu_dev) return fail(BROV_EINVAL, "z0, u, gz0 and gu must not be NULL");
    const size_t need = brov_rollout_vjp_workspace_bytes(e->model, d->n, d->steps);
    if (!d->workspace_dev || d->workspace_bytes < need) return fail(BROV_EINVAL, "workspace too small: need %zu bytes", need);
    memset(a, 0, sizeof(*a));
    int rc = make_consts<double>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a->c);
    if (rc) return rc;
    a->z0 = (const double*)d->z0_dev;
    a->U = (const double*)d->u_dev;
    a->ust = d->u_stride_t; a->usn = d->u_stride_n;
    a->gtraj = (const double*)d->gtraj_dev;
    a->gzT = (const double*)d->gzT_dev;
    a->gz0 = (double*)d->gz0_dev;
    a->gU = (double*)d->gu_dev;
    a->z_out = (double*)d->z_out_dev;
    a->ws = (double*)d->workspace_dev;
    a->health = (unsigned long long*)d->health_dev;
    a->eps = d->singular_eps > 0.0 ? d->singular_eps : 1e-3;
    a->n = d->n;
    a->steps = (int)d->steps;
    a->stride = d->gtraj_dev ? (int)std::min<long long>(d->stride, 0x7fffffffLL) : 1;
    CUDA_TRY(cudaSetDevice(e->device));
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    return BROV_OK;
}

// The refusals every fp64 gradient call starts with, in this order: no engine, a descriptor of the wrong size
// (bad_desc names it; nullptr when the sizes match), a double-integrator engine, an f32 engine, the first-order wrench
// lag.  `what` names the call in the messages.
static int grad_prologue(const brov_engine_t* e, const char* bad_desc, const char* what) {
    if (!e) return fail(BROV_EINVAL, "NULL engine");
    if (bad_desc) return fail(BROV_EINVAL, "%s size mismatch (ABI %d)", bad_desc, BROV_ABI_VERSION);
    if (model_is_di(e->model)) return fail(BROV_EUNSUPPORTED, "%s serves the Fossen models, not double-integrator engines", what);
    if (e->dtype != BROV_F64) return fail(BROV_EUNSUPPORTED, "the gradients are computed in fp64: create the engine with BROV_F64");
    if (e->use_lag1) return fail(BROV_EUNSUPPORTED, "%s does not support the first-order wrench lag", what);
    return BROV_OK;
}

extern "C" int brov_rollout_vjp(brov_engine_t* e, const brov_rollout_vjp_desc* d, void* stream) {
    int rc = grad_prologue(e, !d || d->struct_size != sizeof(brov_rollout_vjp_desc) ? "brov_rollout_vjp_desc" : nullptr,
                           "rollout_vjp");
    if (rc) return rc;
    if (e->pv) return fail(BROV_EUNSUPPORTED, "rollout_vjp uses the shared coefficients: clear the per-vehicle table first");
    AdjArgs a;
    cudaStream_t st = (cudaStream_t)stream;
    rc = rollout_vjp_args(e, d, &a, st);
    if (rc || d->n == 0) return rc;
    CUDA_TRY(launch_adjoint(e->model, d->integrator, a, st));
    return BROV_OK;
}

extern "C" int brov_rollout_vjp_coef(brov_engine_t* e, const brov_rollout_vjp_coef_desc* d, void* stream) {
    const char* bad_desc = !d || d->struct_size != sizeof(brov_rollout_vjp_coef_desc) ? "brov_rollout_vjp_coef_desc"
                           : d->vjp.struct_size != sizeof(brov_rollout_vjp_desc) ? "brov_rollout_vjp_desc" : nullptr;
    int rc = grad_prologue(e, bad_desc, "rollout_vjp");
    if (rc) return rc;
    if (e->pv && e->pv_n != d->vjp.n) return fail(BROV_EINVAL, "vehicle table has %lld rows, call has n = %lld", e->pv_n, d->vjp.n);
    if (d->vjp.n != 0 && !d->gkp_dev) return fail(BROV_EINVAL, "gkp must not be NULL");
    AdjCoefArgs a;
    cudaStream_t st = (cudaStream_t)stream;
    rc = rollout_vjp_args(e, &d->vjp, &a.a, st);
    if (rc || d->vjp.n == 0) return rc;
    a.gkp = (double*)d->gkp_dev;
    a.pv = (const double*)e->pv;
    CUDA_TRY(launch_adjoint_coef(e->model, d->vjp.integrator, a, st));
    return BROV_OK;
}

extern "C" size_t brov_closed_loop_vjp_workspace_bytes(int model, long long n, long long steps) {
    if (model != BROV_THRUSTER8_LAG3 && model != BROV_WRENCH_EULER12 && model != BROV_WRENCH_QUAT13) return 0;
    return cl_adjoint_workspace_bytes(model_nz(model), model_nu(model), n, steps);
}

// no two (step, vehicle) pairs of an operand of E elements addressed at k*st + i*sn + e share an element unless a
// stride is 0 (then the gradient sums them)
static bool cl_strides_disjoint(long long st, long long sn, long long steps, long long n, long long E) {
    if (steps <= 1) st = 0;
    if (n <= 1) sn = 0;
    if (st == 0 && sn == 0) return true;
    if (sn == 0) return st >= E;
    if (st == 0) return sn >= E;
    return (sn >= E && st / sn >= n) || (st >= E && sn / st >= steps);
}

extern "C" int brov_closed_loop_vjp(brov_engine_t* e, const brov_closed_loop_vjp_desc* d, void* stream) {
    int rc = grad_prologue(e, !d || d->struct_size != sizeof(brov_closed_loop_vjp_desc) ? "brov_closed_loop_vjp_desc" : nullptr,
                           "closed_loop_vjp");
    if (rc) return rc;
    rc = cl_check(e, d, 1, d->gtraj_dev != nullptr, "trajectory cotangent", d->gz0_dev, "gz0");
    if (rc || d->n == 0) return rc;
    const int nz = model_nz(e->model), nu = model_nu(e->model);
    struct Op { void* g; long long st, sn; int E; const char* what; } ops[3] = {
        {d->gK_dev, d->K_stride_t, d->K_stride_n, nu * nz, "K"},
        {d->gz_ref_dev, d->z_ref_stride_t, d->z_ref_stride_n, nz, "z_ref"},
        {d->gu_ref_dev, d->u_ref_stride_t, d->u_ref_stride_n, nu, "u_ref"}};
    // the workspace this request needs: z_k, the cotangents of the requested operands, the scratch of a constant one
    unsigned long long per = nz, scr = 0;
    for (int w = 0; w < 3; ++w) {
        if (!ops[w].g) continue;
        if (!cl_strides_disjoint(ops[w].st, ops[w].sn, d->steps, d->n, ops[w].E))
            return fail(BROV_EINVAL, "the gradient of %s needs strides under which distinct (step, vehicle) pairs do not overlap", ops[w].what);
        per += w == 1 ? nz : nu;
        if (ops[w].st == 0 && ops[w].sn == 0) scr = std::max<unsigned long long>(scr, ops[w].E);
    }
    const size_t need = cl_adjoint_bytes(per, scr, d->n, d->steps);    // checked: SIZE_MAX when it does not fit
    if (!d->workspace_dev || d->workspace_bytes < need) return fail(BROV_EINVAL, "workspace too small: need %zu bytes", need);

    ClAdjArgs a;
    memset(&a, 0, sizeof(a));
    if ((rc = make_consts<double>(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &a.c))) return rc;
    cl_operands(e, d, &a);
    a.z0 = (const double*)d->z0_dev;
    a.gtraj = (const double*)d->gtraj_dev;
    a.gzT = (const double*)d->gzT_dev;
    a.gcost = (const double*)d->gcost_dev;
    a.gz0 = (double*)d->gz0_dev;
    a.z_out = (double*)d->z_out_dev;
    double* w = (double*)d->workspace_dev;
    const size_t slab = (size_t)d->n * (size_t)d->steps;
    a.ws = w; w += slab * nz;
    if (d->gK_dev) { a.wgv = w; w += slab * nu; }
    if (d->gz_ref_dev) { a.wgzr = w; w += slab * nz; }
    if (d->gu_ref_dev) { a.wgur = w; w += slab * nu; }
    double* scratch = w;
    a.health = (unsigned long long*)d->health_dev;
    a.n = d->n;
    a.steps = (int)d->steps;
    a.stride = d->gtraj_dev ? (int)std::min<long long>(d->stride, 0x7fffffffLL) : 1;
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d->health_dev) CUDA_TRY(cudaMemsetAsync(d->health_dev, 0, 2 * sizeof(unsigned long long), st));
    CUDA_TRY(launch_closed_loop_adjoint(e->model, d->integrator, a, st));
    for (int o = 0; o < 3; ++o)
        if (ops[o].g) CUDA_TRY(launch_closed_loop_adjoint_reduce(e->model, o, a, (double*)ops[o].g, ops[o].st, ops[o].sn, scratch, st));
    return BROV_OK;
}

// fossen/parameters.py:3-33
template <typename T> static Red9Consts<T> red9_consts() {
    const double m = 11.4, g = 9.82, F_bouy = 1026 * 0.0115 * g;
    const double X_ud = -2.6, Y_vd = -18.5, Z_wd = -13.3, N_rd = -0.28, I_zz = 0.245;
    Red9Consts<T> c;
    c.im_u = (T)(1.0 / (m - X_ud)); c.im_v = (T)(1.0 / (m - Y_vd)); c.im_w = (T)(1.0 / (m - Z_wd)); c.im_r = (T)(1.0 / (I_zz - N_rd));
    c.mYv = (T)(m - Y_vd); c.mXu = (T)(m - X_ud); c.dXY = (T)(X_ud - Y_vd);
    c.Xu = (T)-0.09; c.Xuc = (T)-34.96; c.Yv = (T)-0.26; c.Yvc = (T)-103.25;
    c.Zw = (T)-0.19; c.Zwc = (T)-74.23; c.Nr = (T)-4.64; c.Nrc = (T)-0.43;
    c.wnet = (T)(m * g - F_bouy);
    return c;
}

extern "C" int brov_reduced9_rhs(int dtype, const void* x, const void* u, void* out, long long B, void* stream) {
    if (dtype != BROV_F64 && dtype != BROV_F32) return fail(BROV_EINVAL, "unknown dtype %d", dtype);
    if (B < 0 || B > (long long)0x7fffffff * RED9_BLOCK) return fail(BROV_EINVAL, "B out of range");
    if (B == 0) return BROV_OK;
    if (!x || !u || !out) return fail(BROV_EINVAL, "NULL argument");
    if (dtype == BROV_F32) CUDA_TRY(launch_reduced9<float>(red9_consts<float>(), (const float*)x, (const float*)u, (float*)out, B, (cudaStream_t)stream));
    else CUDA_TRY(launch_reduced9<double>(red9_consts<double>(), (const double*)x, (const double*)u, (double*)out, B, (cudaStream_t)stream));
    return BROV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// host-buffer rollout: time-chunked H2D of inputs on a copy stream, double buffered against the rollout kernels;
// snapshots return on a third stream
// ---------------------------------------------------------------------------------------------------------------
extern "C" int brov_rollout_host(brov_engine_t* e, const brov_rollout_host_desc* d) {
    if (!d || d->struct_size != sizeof(brov_rollout_host_desc)) return fail(BROV_EINVAL, "brov_rollout_host_desc size mismatch (ABI %d)", BROV_ABI_VERSION);
    int rc = check_rollout_common(e, d->integrator, d->n, d->steps, d->dt);
    if (rc) return rc;
    if (d->n == 0) return BROV_OK;
    const bool gen = d->gen.enable != 0;
    if (!d->x0_host || !d->xT_host) return fail(BROV_EINVAL, "x0 and xT must not be NULL");
    if (d->steps > 0 && !d->u_host && !gen) return fail(BROV_EINVAL, "u is NULL");
    if (d->traj_host && d->stride < 1) return fail(BROV_EINVAL, "stride must be >= 1 with a trajectory buffer");
    if (d->lag_in_repr < 0 || d->lag_in_repr > 1 || d->lag_out_repr < 0 || d->lag_out_repr > 1) return fail(BROV_EINVAL, "unknown lag representation");
    CUDA_TRY(cudaSetDevice(e->device));
    const size_t sz = scalar_size(e->dtype);
    const int NX = model_nx(e->model), NU = model_nu(e->model);
    const bool thr = e->model == BROV_THRUSTER8_LAG3;
    const int nl_carry = thr ? 18 : (e->use_lag1 ? 6 : 0);   // what the chunks carry on the device
    const long long n = d->n;
    const size_t row_u = gen ? 0 : (d->u_shared ? 1 : (size_t)n) * NU * sz;  // bytes of one time step of inputs
    const size_t snap_bytes = (size_t)n * NX * sz;
    long long chunk = d->chunk_steps;
    if (chunk <= 0) {
        chunk = gen ? d->steps : (long long)((256ull << 20) / row_u);
        if (d->traj_host) {   // about 256 MiB of snapshots per chunk
            const long long by_traj = d->stride * (long long)std::max<size_t>(1, (256ull << 20) / snap_bytes);
            if (by_traj < chunk) chunk = by_traj;
        }
    }
    if (chunk < 1) chunk = 1;
    if (d->traj_host) chunk = ((chunk + d->stride - 1) / d->stride) * d->stride;  // whole snapshots per chunk
    if (chunk > d->steps) chunk = d->steps > 0 ? d->steps : 1;
    const long long snaps_per_chunk = d->traj_host ? (chunk + d->stride - 1) / d->stride + 1 : 0;

    // per-thruster lag states: wanted back / supplied
    const bool want24 = thr && d->lag_out_host && d->lag_out_repr == BROV_LAG_THRUSTER;
    const bool in24 = thr && d->lag_in_host && d->lag_in_repr == BROV_LAG_THRUSTER;
    long long depth = 0;
    if (want24) {
        if ((rc = carry_depth(e, d->dt, d->integrator == BROV_RK4 ? 4 : 1, &depth))) return rc;
        if (d->lag_in_host && !in24 && d->steps < depth)
            return fail(BROV_EINVAL, "per-thruster lag states cannot be recovered from an allocation-projected lag_in in a call of fewer than %lld steps", depth);
    }

    HostStage& h = e->hs;
    if (!h.ready) {
        CUDA_TRY(cudaStreamCreateWithFlags(&h.s_compute, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&h.s_in, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&h.s_out, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            CUDA_TRY(cudaEventCreateWithFlags(&h.ev_in[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&h.ev_done[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&h.ev_out[b], cudaEventDisableTiming));
        }
        h.ready = true;
    }
    if ((rc = grow(&h.d_x, &h.cap_x, snap_bytes))) return rc;
    if (nl_carry && (rc = grow(&h.d_lag, &h.cap_lag, (size_t)n * nl_carry * sz))) return rc;
    if ((want24 || in24) && (rc = grow(&h.d_lag24, &h.cap_lag24, (size_t)n * 24 * sz))) return rc;
    if (gen && (rc = grow(&h.d_gen, &h.cap_gen, (size_t)n * NU * sz))) return rc;
    if (d->health_host && (rc = grow(&h.d_health, &h.cap_health, 16 + (size_t)n * sz))) return rc;
    if (!gen && d->steps > 0) {
        size_t need_u = (size_t)chunk * row_u, cap = h.cap_u;
        for (int b = 0; b < 2; ++b) { cap = h.cap_u; if ((rc = grow(&h.d_u[b], &cap, need_u))) return rc; }
        h.cap_u = cap;
    }
    if (d->traj_host) {
        size_t need_t = (size_t)snaps_per_chunk * snap_bytes, cap = h.cap_traj;
        for (int b = 0; b < 2; ++b) { cap = h.cap_traj; if ((rc = grow(&h.d_traj[b], &cap, need_t))) return rc; }
        h.cap_traj = cap;
    }

    CUDA_TRY(cudaMemcpyAsync(h.d_x, d->x0_host, snap_bytes, cudaMemcpyHostToDevice, h.s_compute));
    if (nl_carry) {
        if (in24) CUDA_TRY(cudaMemcpyAsync(h.d_lag24, d->lag_in_host, (size_t)n * 24 * sz, cudaMemcpyHostToDevice, h.s_compute));
        else if (d->lag_in_host) CUDA_TRY(cudaMemcpyAsync(h.d_lag, d->lag_in_host, (size_t)n * nl_carry * sz, cudaMemcpyHostToDevice, h.s_compute));
        else CUDA_TRY(cudaMemsetAsync(h.d_lag, 0, (size_t)n * nl_carry * sz, h.s_compute));
    }
    if (gen) {
        if (d->gen.state_in_dev) CUDA_TRY(cudaMemcpyAsync(h.d_gen, d->gen.state_in_dev, (size_t)n * NU * sz, cudaMemcpyHostToDevice, h.s_compute));
        else CUDA_TRY(cudaMemsetAsync(h.d_gen, 0, (size_t)n * NU * sz, h.s_compute));
    }
    if (d->steps == 0 && want24) {   // nothing to integrate: per-thruster states pass through
        if (in24) CUDA_TRY(cudaMemcpyAsync(d->lag_out_host, h.d_lag24, (size_t)n * 24 * sz, cudaMemcpyDeviceToHost, h.s_compute));
        else if (d->lag_in_host) return fail(BROV_EUNSUPPORTED, "a zero-step rollout cannot change the lag representation");
        else memset(d->lag_out_host, 0, (size_t)n * 24 * sz);
    }
    long long done = 0;
    int b = 0;
    bool tail_started = false;
    for (long long c = 0; done < d->steps; ++c, b ^= 1) {
        const long long len = (d->steps - done < chunk) ? (d->steps - done) : chunk;
        if (!gen) {
            // inputs of chunk c -> d_u[b] once the kernel that last read d_u[b] (chunk c-2) has finished
            if (c >= 2) CUDA_TRY(cudaStreamWaitEvent(h.s_in, h.ev_done[b], 0));
            CUDA_TRY(cudaMemcpyAsync(h.d_u[b], (const char*)d->u_host + (size_t)done * row_u, (size_t)len * row_u, cudaMemcpyHostToDevice, h.s_in));
            CUDA_TRY(cudaEventRecord(h.ev_in[b], h.s_in));
            CUDA_TRY(cudaStreamWaitEvent(h.s_compute, h.ev_in[b], 0));
        }
        const long long first_snap = d->traj_host ? done / d->stride : 0;
        const long long last_snap = d->traj_host ? (done + len) / d->stride : 0;  // snapshots [first, last)
        if (d->traj_host && c >= 2) CUDA_TRY(cudaStreamWaitEvent(h.s_compute, h.ev_out[b], 0));
        brov_rollout_desc r;
        memset(&r, 0, sizeof(r));
        r.struct_size = sizeof(r);
        r.integrator = d->integrator; r.n = n; r.steps = len; r.dt = d->dt;
        r.x0_dev = h.d_x; r.xT_dev = h.d_x; r.u_dev = gen ? nullptr : h.d_u[b];
        r.u_stride_t = d->u_shared ? NU : n * NU;
        r.u_stride_n = d->u_shared ? 0 : NU;
        // chunk 0 reads the caller's lag in its own representation; every chunk leaves the projected lag in d_lag
        const bool first24 = c == 0 && in24;
        r.lag_in_dev = nl_carry ? (first24 ? h.d_lag24 : h.d_lag) : nullptr;
        r.lag_in_repr = first24 ? BROV_LAG_THRUSTER : BROV_LAG_PROJECTED;
        r.lag_out_dev = nl_carry ? h.d_lag : nullptr;
        r.lag_out_repr = BROV_LAG_PROJECTED;
        r.traj_dev = d->traj_host ? h.d_traj[b] : nullptr;
        r.stride = d->traj_host ? d->stride : 1; r.step0 = done; r.snap_base = first_snap;
        r.time_slices = 0;
        if (gen) {
            r.gen = d->gen;
            r.gen.state_in_dev = h.d_gen; r.gen.state_out_dev = h.d_gen;
        }
        if (d->health_host) {
            r.health_dev = h.d_health;
            r.min_abs_cos_dev = (char*)h.d_health + 16;
            r.min_abs_cos_accumulate = c > 0;
            r.singular_eps = d->singular_eps;
        }
        // per-thruster states: rebuilt by the chunks that cover the last `depth` steps of the call
        Lag24 l24 = {nullptr, nullptr, true};
        if (want24 && done + len > d->steps - depth) {
            l24.out = h.d_lag24;
            l24.in = (tail_started || (done == 0 && in24)) ? h.d_lag24 : nullptr;
            tail_started = true;
        }
        rc = e->dtype == BROV_F32 ? rollout_impl<float>(e, &r, h.s_compute, l24) : rollout_impl<double>(e, &r, h.s_compute, l24);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(h.ev_done[b], h.s_compute));
        if (d->traj_host && last_snap > first_snap) {
            CUDA_TRY(cudaStreamWaitEvent(h.s_out, h.ev_done[b], 0));
            CUDA_TRY(cudaMemcpyAsync((char*)d->traj_host + (size_t)first_snap * snap_bytes, h.d_traj[b], (size_t)(last_snap - first_snap) * snap_bytes, cudaMemcpyDeviceToHost, h.s_out));
        }
        if (d->traj_host) CUDA_TRY(cudaEventRecord(h.ev_out[b], h.s_out));
        done += len;
    }
    CUDA_TRY(cudaMemcpyAsync(d->xT_host, h.d_x, snap_bytes, cudaMemcpyDeviceToHost, h.s_compute));
    if (nl_carry && d->lag_out_host && d->steps > 0) {
        if (want24) CUDA_TRY(cudaMemcpyAsync(d->lag_out_host, h.d_lag24, (size_t)n * 24 * sz, cudaMemcpyDeviceToHost, h.s_compute));
        else CUDA_TRY(cudaMemcpyAsync(d->lag_out_host, h.d_lag, (size_t)n * nl_carry * sz, cudaMemcpyDeviceToHost, h.s_compute));
    } else if (nl_carry && d->lag_out_host && !want24) {
        CUDA_TRY(cudaMemcpyAsync(d->lag_out_host, h.d_lag, (size_t)n * nl_carry * sz, cudaMemcpyDeviceToHost, h.s_compute));
    }
    if (gen && d->gen.state_out_dev) CUDA_TRY(cudaMemcpyAsync(d->gen.state_out_dev, h.d_gen, (size_t)n * NU * sz, cudaMemcpyDeviceToHost, h.s_compute));
    if (d->health_host) {
        if (d->steps > 0) CUDA_TRY(cudaMemcpyAsync(d->health_host, h.d_health, 16, cudaMemcpyDeviceToHost, h.s_compute));
        else { d->health_host[0] = 0; d->health_host[1] = 0; }
    }
    CUDA_TRY(cudaStreamSynchronize(h.s_in));
    CUDA_TRY(cudaStreamSynchronize(h.s_compute));
    CUDA_TRY(cudaStreamSynchronize(h.s_out));
    return BROV_OK;
}

extern "C" int brov_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(BROV_EINVAL, "out is NULL");
    CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return BROV_OK;
}
extern "C" int brov_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return BROV_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// FP pipe peak
// ---------------------------------------------------------------------------------------------------------------
extern "C" int brov_fma_peak(int dtype, int device, int iters, double* tflops_out, double* ms_out) {
    if (dtype != BROV_F64 && dtype != BROV_F32) return fail(BROV_EINVAL, "unknown dtype %d", dtype);
    if (iters < 1) return fail(BROV_EINVAL, "iters must be >= 1");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8;
    void* scratch = nullptr;
    CUDA_TRY(cudaMalloc(&scratch, (size_t)blocks * 256 * 8));
    cudaEvent_t t0, t1;
    CUDA_TRY(cudaEventCreate(&t0));
    CUDA_TRY(cudaEventCreate(&t1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CUDA_TRY(cudaEventRecord(t0, 0));
        if (dtype == BROV_F32) CUDA_TRY(launch_fma_peak<float>(iters, blocks, (float*)scratch, 0));
        else CUDA_TRY(launch_fma_peak<double>(iters, blocks, (double*)scratch, 0));
        CUDA_TRY(cudaEventRecord(t1, 0));
        CUDA_TRY(cudaEventSynchronize(t1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, t0, t1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(scratch);
    const double flops = (double)blocks * 256.0 * (double)iters * 64.0 * 2.0;
    if (tflops_out) *tflops_out = flops / (best * 1e-3) / 1e12;
    if (ms_out) *ms_out = best;
    return BROV_OK;
}
