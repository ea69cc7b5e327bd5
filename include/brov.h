/* brov.h — C ABI of libbrov.so, the B200 (sm_100a) batched BlueROV2 Fossen-dynamics engine.
 *
 * This is the drop-in boundary for the reference's hot path.  The reference (ViktorNfa/bluerov2_dynamics) is pure
 * Python and has no FFI layer; what it offers instead is a Python call surface, and each entry point below is what
 * a binding of that surface calls (the ctypes stub a maintainer would add is shown in INTEGRATION.md and lives in
 * bluerov2_dynamics_b200/_lib.py).  Citations are file:line in the reference checkout.
 *
 * Conventions
 *   - plain C types only; every array is row-major and contiguous; "dev" pointers are device pointers valid in the
 *     calling process's primary CUDA context on the engine's device, "host" pointers are host pointers;
 *   - arrays have the engine's scalar type (float for BROV_F32, double for BROV_F64) unless typed otherwise;
 *   - every call returns 0 on success, a negative BROV_E* code otherwise; brov_last_error() describes the last
 *     failure on the calling thread;
 *   - device calls are asynchronous on `stream` (a cudaStream_t cast to void*; NULL = legacy default stream);
 *   - an engine handle is not thread-safe; use one per stream.
 *
 * State layouts (same as the reference)
 *   BROV_THRUSTER8_LAG3  x[12] = [x y z phi theta psi u v w p q r], input u[8] = normalised thruster voltages,
 *                        hidden lag state lag[8][3] (ThrusterLag._x of each thruster)     fossen/BlueROV2.py:357-400
 *   BROV_WRENCH_EULER12  x[12] as above, input tau[6] = body wrench                    fossen/BlueROV2_thrust.py:235
 *   BROV_WRENCH_QUAT13   x[13] = [x y z qw qx qy qz u v w p q r], input tau[6]         fossen/BlueROV2_wrench.py:322
 *   With the optional first-order wrench lag enabled (extension, no reference counterpart) the two wrench models
 *   carry a hidden state lag[6] = filtered wrench.
 */
#ifndef BROV_H
#define BROV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BROV_ABI_VERSION 8

enum { BROV_THRUSTER8_LAG3 = 0, BROV_WRENCH_EULER12 = 1, BROV_WRENCH_QUAT13 = 2,
       /* double-integrator comparison model of the reference's evaluation tables (kinematics + a learned linear map
        * input -> body accelerations); every rollout / evaluator entry point below serves it as well:
        *   simulate_double_integrator / multistep_rmse_endpoint_di
        *   RK4, 8 thruster inputs        training/train_tank_brov2_rk4.py:461-547
        *   Euler, 8 thruster inputs      training/train_tank_brov2_full_comparison.py:531-598
        *   Euler, 6 wrench inputs        training/train_tank_brov2_wrench_comp.py:293-366
        *   quaternion Euler, 6 inputs    training/train_tank_brov2_wrench_quat.py:324-397 */
       BROV_DI_EULER12_U8 = 3, BROV_DI_EULER12_U6 = 4, BROV_DI_QUAT13_U6 = 5 };
enum { BROV_F64 = 0, BROV_F32 = 1 };
enum { BROV_RK4 = 0, BROV_EULER = 1 };
/* representation of the thruster model's hidden lag state in lag_in / lag_out arrays */
enum { BROV_LAG_THRUSTER = 0,   /* [n][8][3]: ThrusterLag._x of each thruster (the reference's hidden state) */
       BROV_LAG_PROJECTED = 1 }; /* [n][6][3]: Z_c = sum_i alloc[c][i] * lag_i — see below */

enum {
    BROV_OK = 0,
    BROV_EINVAL = -1,   /* bad argument */
    BROV_ECUDA = -2,    /* CUDA runtime error (text in brov_last_error) */
    BROV_ENOMEM = -3,
    BROV_EUNSUPPORTED = -4
};

/* Physical parameter vector (double[BROV_NPHYS]): the scalar attributes of the reference classes
 * (fossen/BlueROV2.py:81-150 = BlueROV2_thrust.py:82-147 = BlueROV2_wrench.py:160-225). */
enum {
    BROV_PH_M = 0, BROV_PH_W = 1, BROV_PH_B = 2,
    BROV_PH_XB = 3, /* xb yb zb */
    BROV_PH_I = 6,  /* Ix Iy Iz */
    BROV_PH_ADDED = 9,   /* Xu_dot Yv_dot Zw_dot Kp_dot Mq_dot Nr_dot */
    BROV_PH_LIN = 15,    /* Xu Yv Zw Kp Mq Nr */
    BROV_PH_QUAD = 21,   /* Xu_abs ... Nr_abs */
    BROV_PH_MINV = 27,   /* diag(Minv): kept separate because the reference freezes Minv in __init__ (trap T5) */
    BROV_PH_CURRENT = 33,/* current_speed, NED */
    BROV_PH_TLAG1 = 36,  /* first-order wrench lag time constant [s] (extension) */
    BROV_NPHYS = 37
};
/* Kernel coefficient vector (double[BROV_NKP]) derived from the physical one; layout in csrc/brov_device.cuh. */
#define BROV_NKP 36
#define BROV_MAX_H 4

typedef struct brov_engine brov_engine_t;

int brov_abi_version(void);
const char* brov_last_error(void);

/* Engine lifetime.  Replaces `BlueROV2(rho=..., current_speed=...)` (fossen/BlueROV2.py:79): the new engine holds
 * the reference constants, the reference thruster geometry and the reference lag model. */
int brov_create(int model, int dtype, int device, brov_engine_t** out);
void brov_destroy(brov_engine_t* e);

/* Constants. */
int brov_default_physical(double rho, double* phys /*[BROV_NPHYS]*/);          /* fossen/BlueROV2.py:81-150 */
int brov_derive_params(const double* phys /*[BROV_NPHYS]*/, double* kp /*[BROV_NKP]*/);
int brov_default_allocation(double* alloc /*[6][8]*/, double* r /*[8][3] or NULL*/, double* dir /*[8][3] or NULL*/);
                                                                                /* fossen/BlueROV2.py:159-232 */
int brov_set_params(brov_engine_t* e, const double* kp /*[BROV_NKP]*/);
int brov_get_params(const brov_engine_t* e, double* kp /*[BROV_NKP]*/);
int brov_set_allocation(brov_engine_t* e, const double* alloc /*[6][8]*/);
/* Gains of a BROV_DI_* engine as estimate_di_gains returns them (training/train_tank_brov2_rk4.py:438-458):
 * v_dot = u K_lin, w_dot = u K_ang; K_lin, K_ang are [NU][3] row-major, NU = 8 or 6 by engine model. */
int brov_set_di_gains(brov_engine_t* e, const double* K_lin, const double* K_ang);
/* Per-vehicle (Monte-Carlo) coefficient table, dev, engine scalar type, layout [BROV_NKP][n]; NULL clears it.
 * The table is borrowed, not copied: it must outlive the calls that use it.  any_current: non-zero if some row has a
 * non-zero ocean current (rows KP 31..33); zero lets the kernels skip the relative-velocity terms. */
int brov_set_vehicle_params(brov_engine_t* e, const void* kp_soa_dev, long long n, int any_current);
/* Optional first-order wrench lag tau_dot = (tau_cmd - tau)/T_lag for the two wrench models (extension). */
int brov_set_wrench_lag1(brov_engine_t* e, int enable);

/* ThrusterLag discretisation (fossen/BlueROV2.py:490-501: scipy cont2discrete(zoh)).  `discretize` computes the
 * zero-order hold natively (matrix exponential, extended precision); `set_lag_discrete` overrides (Ad, Bd) for one
 * dt, e.g. with scipy's own result. */
int brov_lag_discretize(double dt, double* Ad /*[3][3]*/, double* Bd /*[3]*/);
int brov_set_lag_discrete(brov_engine_t* e, double dt, const double* Ad, const double* Bd);

/* One state-derivative evaluation for n vehicles — `rov.dynamics(x, u, dt)` (fossen/BlueROV2.py:357,
 * BlueROV2_thrust.py:235, BlueROV2_wrench.py:322).  x [n][NX], u [n][NU], xdot [n][NX] (NX+6 with the wrench lag:
 * the last 6 are tau_dot).  lag_inout [n][NLAG] or NULL: for the thruster model the lag state is read, advanced by
 * ONE ThrusterLag.step and written back, exactly as a reference dynamics() call mutates it (NULL = zero state,
 * nothing written). */
int brov_rhs(brov_engine_t* e, long long n, const void* x_dev, const void* u_dev, void* lag_inout_dev, double dt,
             void* xdot_dev, void* stream);

/* Thruster map alone — `rov.compute_thruster_forces(u_thrust, dt)` (fossen/BlueROV2.py:265-278): voltages -> T200
 * polynomial -> ONE ThrusterLag.step per thruster -> body wrench.  u [n][8], lag_inout [n][8][3] or NULL (zero state,
 * nothing written), tau [n][6].  BROV_THRUSTER8_LAG3 engines only. */
int brov_thruster_wrench(brov_engine_t* e, long long n, const void* u_dev, void* lag_inout_dev, double dt,
                         void* tau_dev, void* stream);

/* Thruster map along a recorded input series with ONE carried lag state — the loop
 * `[rov.compute_thruster_forces(u, dt) for u in U]` (make_pinc_dataset, training/train_tank_brov2_rk4.py:676-696) as one
 * launch: u [rows][8], tau [rows][6]; lag0 [8][3] = lag state before row 0 or NULL (zeros); lag_end [8][3] = state after
 * the last row or NULL.  Rows are evaluated in parallel by replaying, per row, the tail of the input history that the
 * stable lag filter still remembers (brov_se_carry_steps(e, dt, BROV_EULER) rows). */
int brov_thruster_wrench_series(brov_engine_t* e, long long rows, const void* u_dev, const void* lag0_dev, double dt,
                                void* tau_dev, void* lag_end_dev, void* stream);

/* The same two calls with every array in HOST memory (engine scalar type): what a model object's `dynamics()` /
 * `compute_thruster_forces()` costs per call is launch latency, so inputs and outputs travel in one pinned staging
 * buffer each way and the call returns after the results have landed.  lag_inout_host as above ([n][8][3] or NULL). */
int brov_rhs_host(brov_engine_t* e, long long n, const void* x_host, const void* u_host, void* lag_inout_host,
                  double dt, void* xdot_host);
int brov_thruster_wrench_host(brov_engine_t* e, long long n, const void* u_host, void* lag_inout_host, double dt,
                              void* tau_host);

/* Open-loop rollout — `simulate_physics(x0, U_seq, dt, rov)` for n vehicles at once
 * (RK4: training/train_tank_brov2_rk4.py:375-396; Euler: training/train_tank_brov2_full_comparison.py:453-466,
 * quaternion re-normalisation per step: training/train_tank_brov2_wrench_quat.py:262-263).
 * Input element (step k, vehicle i, channel j) is read at u[k*u_stride_t + i*u_stride_n + j] (strides in scalars):
 *   per-vehicle series, time-major  [steps][n][NU] : u_stride_t = n*NU, u_stride_n = NU
 *   one series shared by all        [steps][NU]    : u_stride_t = NU,   u_stride_n = 0
 *   one constant input per vehicle  [n][NU]        : u_stride_t = 0,    u_stride_n = NU
 * With an RK4 step the thruster lag advances four times per step (once per stage) as in the reference.
 * Lag representation.  The eight thruster lags are copies of one linear filter, so the six allocation-projected
 * combinations Z_c = sum_i alloc[c][i] lag_i obey the same recurrence driven by (alloc F)_c and yield the identical
 * wrench with 18 instead of 24 hidden values and ~150 fewer operations per RK4 step.  Every rollout integrates in that
 * form.  lag_out_repr = BROV_LAG_PROJECTED returns Z ([n][6][3], a valid lag_in with lag_in_repr = BROV_LAG_PROJECTED
 * for the next chunk, and the cheapest carry).  lag_out_repr = BROV_LAG_THRUSTER (the default, the reference's hidden
 * state ThrusterLag._x, fossen/BlueROV2.py:503-510) is produced by a short second kernel: each thruster's lag is a
 * stable linear filter of that thruster's input alone, so its state after the call is fixed — to below one ulp — by
 * the last brov_se_carry_steps(e, dt, integrator) inputs of the call (or by lag_in and all inputs of a shorter call);
 * one thread per (vehicle, thruster) replays them.  A projected lag_in with a per-thruster lag_out is therefore only
 * accepted when the call is at least that many steps long.
 * traj (optional): state after global step g = step0+k+1 is stored when g % stride == 0, as snapshot
 * s = g/stride - 1 at traj[(s - snap_base)][n][NX].  Chunked rollouts pass xT/lag_out of one call as x0/lag_in of
 * the next and advance step0.
 *
 * Generated inputs (gen.enable != 0): the input of every step is produced inside the kernel instead of being read
 * from u_dev — the reference's smooth random command signal (training/train_sim_brov2_koopmanEDMDc.py:161-164,180)
 *     s_k = clip(rho s_{k-1} + sigma N(0,1), -clip, clip),   u_k[j] = scale[j] s_k[j],   s_{-1} = state_in (or 0)
 * with N(0,1) from the counter-based generator Philox4x32-10 keyed on `seed` at counter (vehicle0 + i, step0 + k):
 * chunked, sliced and sharded rollouts see the same stream, nothing is read from HBM per step.  The AR(1) state
 * ([n][NU], in units of u) is the only thing carried (state_in_dev / state_out_dev).  brov_generate_inputs
 * materialises the same signal for a subset of vehicles so that a CPU reference can consume identical inputs.
 *
 * Health accounting (optional): health_dev (unsigned long long[2], dev) receives the number of vehicles whose final
 * state holds a non-finite value and the number whose |cos theta| came below singular_eps at the start of some step
 * — the singularity of the Euler-angle kinematics, where the reference clamps cos theta (fossen/BlueROV2.py:52-56) and
 * amplifies rounding differences without bound.  min_abs_cos_dev ([n], engine scalar type) holds the running minimum
 * of |cos theta| per vehicle: with min_abs_cos_accumulate != 0 the incoming values are kept (chunked rollouts),
 * otherwise the call starts from 1.  Quaternion and double-integrator models report 1 / zero counts. */
typedef struct brov_input_gen {
    int32_t enable;
    int32_t reserved;
    uint64_t seed;
    long long vehicle0;         /* global index of local vehicle 0: key of the random stream (sharded ensembles) */
    double rho, sigma, clip;    /* reference: 0.98, 0.02, 1.0 */
    double scale[8];            /* per input channel; the reference drives all thrusters with scale 1 */
    const void* state_in_dev;   /* [n][NU] engine scalar type, or NULL = zeros */
    void* state_out_dev;        /* [n][NU] or NULL (may alias state_in_dev) */
} brov_input_gen;

typedef struct brov_rollout_desc {
    uint32_t struct_size;       /* = sizeof(brov_rollout_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* x0_dev;         /* [n][NX] */
    void* xT_dev;               /* [n][NX], may alias x0_dev */
    const void* u_dev;          /* ignored with generated inputs */
    long long u_stride_t, u_stride_n;
    const void* lag_in_dev;     /* [n][NLAG] or NULL = zeros */
    void* lag_out_dev;          /* [n][NLAG] or NULL (may alias lag_in_dev when the representations agree) */
    void* traj_dev;             /* or NULL */
    long long stride;           /* >= 1 when traj_dev != NULL */
    long long step0;
    long long snap_base;
    int32_t lag_in_repr;        /* BROV_LAG_* (thruster model only) */
    int32_t lag_out_repr;
    /* Temporal tiling of the launch (results are bit-identical for every value): 0 = automatic, 1 = off, Q > 1 = cut
     * the steps of this call into Q slices per block of vehicles.  Vehicles are independent, but B vehicle blocks on S
     * resident slots cost ceil(B/S) rounds of the full step count; slicing makes it ceil(B*Q/S) rounds of steps/Q
     * (cfg2: 512 blocks on 296 slots, Q = 4 -> 7 rounds of 25 steps instead of 2 rounds of 100).  Slices of one
     * vehicle block hand their state over through xT and engine-owned scratch. */
    int32_t time_slices;
    int32_t min_abs_cos_accumulate;
    void* health_dev;           /* unsigned long long[2] or NULL */
    void* min_abs_cos_dev;      /* [n] or NULL */
    double singular_eps;        /* 0 = 1e-3 */
    brov_input_gen gen;
} brov_rollout_desc;
int brov_rollout(brov_engine_t* e, const brov_rollout_desc* d, void* stream);

/* The generated command signal as an array: out [steps][n_sel][nu] holds the inputs of steps step0 .. step0+steps-1
 * for the selected vehicles first, first + vstride, ..., first + (n_sel-1) vstride (local indices; the stream key is
 * gen.vehicle0 + index).  gen.state_in_dev / state_out_dev are [n_sel][nu] arrays indexed by selected vehicle.  Same
 * device code as the rollout kernels: a rollout fed with `out` reproduces the generated-input rollout bit for bit. */
typedef struct brov_gen_inputs_desc {
    uint32_t struct_size;
    int32_t dtype;              /* BROV_F64 / BROV_F32 */
    int32_t nu;                 /* 8 or 6 */
    int32_t device;
    long long first, vstride, n_sel;
    long long step0, steps;
    brov_input_gen gen;
    void* out_dev;
} brov_gen_inputs_desc;
int brov_generate_inputs(const brov_gen_inputs_desc* d, void* stream);
/* One integrator step with one input row per vehicle (u [n][NU]) — the body of the reference's simulate_physics loop
 * as a call; lag_inout [n][NLAG] or NULL (zero lag, nothing written).  x_out may alias x. */
int brov_step(brov_engine_t* e, int integrator, long long n, const void* x_dev, const void* u_dev, double dt,
              void* x_out_dev, void* lag_inout_dev, void* stream);

/* Multi-step endpoint squared error over sliding windows — `multistep_rmse_endpoint_physics(X, U, H, dt)`
 * (training/train_tank_brov2_rk4.py:399-417 and the Euler twins in train_tank_brov2_full_comparison.py:469-487,
 * train_tank_brov2_wrench_comp.py:232-250, train_tank_brov2_wrench_quat.py:279-297) for up to BROV_MAX_H horizons in
 * one pass; with H = {1} and BROV_EULER it is also `one_step_rmse_physics`.
 * X [rows][NX], U [rows][NU]: one recorded series.  Window k in [0, n_windows) starts at X[k] and is driven by
 * U[k..]; it contributes to horizon H_h iff k + H_h <= rows-1.  se_out_dev[h] (double[BROV_MAX_H], dev) receives the
 * sum over windows of |x_end - X[k+H_h]|^2; count_out[h] (host, may be NULL) the number of contributing windows;
 * rmse_h = sqrt(se_h / (count_h * NX)).  lag0_dev [n_windows][24] or NULL: initial lag state per window (the
 * reference shares ONE model object over all windows so its lag state leaks from window to window, SURVEY trap T3;
 * this evaluator is window-parallel and starts each window from lag0, default zero).
 * workspace_dev: at least brov_se_workspace_bytes(n_windows) bytes. */
typedef struct brov_se_desc {
    uint32_t struct_size;
    int32_t integrator;
    long long rows;
    long long n_windows;
    double dt;
    const void* X_dev;
    const void* U_dev;
    const void* lag0_dev;
    int32_t n_horizons;
    int32_t horizons[BROV_MAX_H];   /* strictly ascending, >= 1 */
    double* se_out_dev;             /* [BROV_MAX_H] */
    long long* count_out;           /* host [BROV_MAX_H] or NULL */
    void* workspace_dev;
    size_t workspace_bytes;
    /* lag_carry != 0 (thruster model, n_horizons must be 1, lag0_dev must be NULL): reproduce the reference's literal
     * behaviour — ONE model object scores all windows in order, so window k starts from the lag state left by windows
     * 0..k-1 (each feeding U[w..w+H-1], every step advancing the lag 4x under RK4, 1x under Euler).  The lag is a
     * stable linear filter of the inputs only; each window replays the tail of that history that is distinguishable
     * from zero in floating point (about 45 RK4 / 180 Euler steps), so windows stay independent and the result agrees
     * with the sequential reference to rounding.  window0 / row0: global indices of local window 0 and local row 0
     * when the series is a shard (rows before the shard's first window must then be present back to the replay depth,
     * brov_se_carry_rows). */
    int32_t lag_carry;
    /* time slices of the longest horizon (reset mode): 0 = automatic (against the partial last wave of window blocks,
     * as brov_rollout_desc.time_slices), 1 = off, 2..4 forced.  The per-window results do not depend on it; the
     * squared-error sums are added in another order (agreement to rounding, bit-reproducible for a given value). */
    int32_t time_slices;
    long long window0;
    long long row0;
    /* optional health accounting as in brov_rollout_desc: windows whose endpoint error is not finite / that came within
     * singular_eps of the Euler-angle singularity (unsigned long long[2], dev; zeroed by the call) */
    void* health_dev;
    double singular_eps;        /* 0 = 1e-3 */
} brov_se_desc;
/* Number of integrator steps of history a carried-lag window replays for this dt / integrator (also the number of
 * rows a shard must hold before its first window, plus one). */
int brov_se_carry_steps(brov_engine_t* e, double dt, int integrator, long long* steps_out);
size_t brov_se_workspace_bytes(long long n_windows);
int brov_multistep_se(brov_engine_t* e, const brov_se_desc* d, void* stream);

/* Candidate sweep of the evaluator: the squared-error sums of brov_multistep_se for n_candidates coefficient sets
 * against ONE recorded series, in one launch — calibration of the uncertain hydrodynamic coefficients against a tank
 * recording, sensitivity studies, scoring a Monte-Carlo cloud of vehicles.  Fossen models only (thruster8, wrench12,
 * quat13); the first-order wrench lag is not supported.
 * kp_soa_dev: [BROV_NKP][n_candidates], engine scalar type, the layout of brov_set_vehicle_params (candidate c is
 * column c); any_current: non-zero if some candidate has a non-zero ocean current.  The table travels in the
 * descriptor: the engine's shared coefficients and its per-vehicle table are neither used nor changed.  Allocation and
 * lag discretisation come from the engine.
 * se_out_dev [n_candidates][BROV_MAX_H] (double, dev): row c is what brov_multistep_se(time_slices = 1) returns with
 * candidate c's coefficients (the same per-window arithmetic and summation order); count_out (host, may be NULL) is the
 * same for every candidate.  health_dev [n_candidates][2] (unsigned long long, dev) or NULL: per candidate, the windows
 * with a non-finite endpoint error / that came within singular_eps of theta = +-pi/2 (zeroed by the call).
 * Geometry fields (integrator ... lag_carry, window0, row0) as in brov_se_desc.  lag_carry: the lag state each window
 * inherits does not depend on the coefficients, so one pre-pass computes it for all candidates.  workspace_dev: at least
 * brov_se_sweep_workspace_bytes(n_candidates, n_windows, lag_carry) bytes.  n_candidates * ceil(n_windows / 128) must
 * stay below 2^31 (split larger sweeps into several calls). */
typedef struct brov_se_sweep_desc {
    uint32_t struct_size;
    int32_t integrator;
    long long rows;
    long long n_windows;
    double dt;
    const void* X_dev;
    const void* U_dev;
    const void* lag0_dev;           /* [n_windows][24] or NULL, shared by all candidates (reset mode) */
    int32_t n_horizons;
    int32_t horizons[BROV_MAX_H];
    int32_t lag_carry;
    long long window0;
    long long row0;
    long long n_candidates;
    const void* kp_soa_dev;         /* [BROV_NKP][n_candidates] */
    int32_t any_current;
    int32_t reserved;
    double* se_out_dev;             /* [n_candidates][BROV_MAX_H] */
    long long* count_out;           /* host [BROV_MAX_H] or NULL */
    void* health_dev;               /* [n_candidates][2] or NULL */
    double singular_eps;            /* 0 = 1e-3 */
    void* workspace_dev;
    size_t workspace_bytes;
} brov_se_sweep_desc;
size_t brov_se_sweep_workspace_bytes(long long n_candidates, long long n_windows, int lag_carry);
int brov_multistep_se_sweep(brov_engine_t* e, const brov_se_sweep_desc* d, void* stream);

/* Exact derivatives of the evaluator's squared-error sums in the coefficients — what a least-squares calibration of the
 * hydrodynamic coefficients against a recorded series needs.  With r_w the endpoint residual of window w at horizon
 * H_h and J_w = d x_end / d theta its sensitivity (forward mode, propagated through the integrator steps):
 *     se_out_dev[h]          = sum_w |r_w|^2                 (brov_multistep_se's sum, to rounding)
 *     grad_out_dev[h][j]     = sum_w 2 r_w . J_w[:, j]       (d se_h / d theta_j)
 *     gn_out_dev[h][i][j]    = sum_w J_w[:, i] . J_w[:, j]   (Gauss-Newton matrix; exactly symmetric)
 * theta is a point of n_dirs parameters given through the coefficient vector it maps to: kp_dev [BROV_NKP] (double,
 * dev) is the point, row j of dirs_dev [n_dirs][BROV_NKP] (double, dev) is d kp / d theta_j — any directions, so the
 * call knows nothing about physical parameters (bluerov2_dynamics_b200.engine.coefficient_directions builds them from
 * the physical vector).  The engine's own coefficients are neither used nor changed; allocation and lag
 * discretisation come from the engine.  any_current: non-zero if kp has an ocean current or some direction moves it.
 * The derivative is that of the computed function, branch taken: d|x| = sign(x) dx, the clamped cos(theta) and the
 * quaternion fallback have zero derivative.  The thruster map and its lag do not depend on the coefficients.
 * fp64 engines, Fossen models (thruster8, wrench12, quat13), RK4 / Euler; f32 engines, double-integrator engines and
 * the first-order wrench lag return BROV_EUNSUPPORTED; 1 <= n_dirs <= BROV_NKP.  Geometry fields (integrator ...
 * lag_carry, window0, row0), count_out and the health counters (unsigned long long[2], dev, zeroed by the call) as in
 * brov_se_desc.  The sums are added in a fixed order: bit-reproducible run to run.  workspace_dev: at least
 * brov_se_grad_workspace_bytes(n_windows, n_dirs, lag_carry) bytes; it does not grow with n_windows except for the
 * carried lag ([n_windows][18]). */
typedef struct brov_se_grad_desc {
    uint32_t struct_size;
    int32_t integrator;
    long long rows;
    long long n_windows;
    double dt;
    const void* X_dev;
    const void* U_dev;
    const void* lag0_dev;           /* [n_windows][24] or NULL (reset mode) */
    int32_t n_horizons;
    int32_t horizons[BROV_MAX_H];
    int32_t lag_carry;
    long long window0;
    long long row0;
    const double* kp_dev;           /* [BROV_NKP] */
    int32_t any_current;
    int32_t n_dirs;
    const double* dirs_dev;         /* [n_dirs][BROV_NKP] */
    double* se_out_dev;             /* [BROV_MAX_H] */
    double* grad_out_dev;           /* [BROV_MAX_H][n_dirs] */
    double* gn_out_dev;             /* [BROV_MAX_H][n_dirs][n_dirs] */
    long long* count_out;           /* host [BROV_MAX_H] or NULL */
    void* health_dev;               /* [2] or NULL */
    double singular_eps;            /* 0 = 1e-3 */
    void* workspace_dev;
    size_t workspace_bytes;
} brov_se_grad_desc;
size_t brov_se_grad_workspace_bytes(long long n_windows, int n_dirs, int lag_carry);
int brov_multistep_se_grad(brov_engine_t* e, const brov_se_grad_desc* d, void* stream);

/* Exact Jacobians of every integrator step along batched trajectories — what LQR / MPC about a trim point, iLQR about
 * a nominal trajectory or an EKF needs.  With Phi the discrete step of the engine (integrator, dt),
 *     z_{k+1} = Phi(z_k, u_k),   jac_dev[k][i] = J_k = [A_k | B_k] = [dPhi/dz | dPhi/du] (z_k, u_k)   for vehicle i.
 * z is the full state the step depends on: z = [x (NX) | Z (18, thruster model only)], with Z[c][k] (c = 0..5, k = 0..2)
 * the allocation-projected lag (BROV_LAG_PROJECTED, see brov_rollout_desc) in that [6][3] order.  NZ = 30 / 12 / 13 and
 * NU = 8 / 6 / 6 for thruster8 / wrench12 / quat13; J has NC = NZ + NU columns, state columns first, then the inputs.
 * Jacobians in per-thruster lag coordinates L [8][3] follow by the chain rule with Z = P L (P = alloc per lag
 * component); they are rank-deficient there, since the dynamics see L only through Z.
 * The derivative is that of the computed function, branch taken (as brov_multistep_se_grad): d|x| = sign(x) dx, the
 * clamped cos(theta) and the quaternion fallback are constants.  Every stage evaluates full sines and cosines, so the
 * primal z agrees with brov_rollout to rounding, not bit for bit.  The lag rows are closed form: dZ'/dx = 0,
 * dZ'/dZ = lagA per channel, dZ'/du_i = lagB (x) alloc[:, i] F'(u_i) with F the T200 curve.
 * The engine's shared coefficients (brov_set_params), allocation and lag discretisation for dt (brov_set_lag_discrete
 * overrides apply) are used.  fp64 engines, Fossen models, RK4 / Euler; f32 engines, double-integrator engines, the
 * first-order wrench lag and an engine with a per-vehicle coefficient table (clear it first) return
 * BROV_EUNSUPPORTED.  steps >= 1; n = 0 is a no-op.
 *   z0_dev [n][NZ]; u_dev with u_stride_t / u_stride_n as in brov_rollout_desc (per-vehicle, shared or constant);
 *   z_out_dev [n][NZ] or NULL: z after the last step (may alias z0_dev);
 *   z_traj_dev [steps][n][NZ] or NULL: z after every step;
 *   jac_dev [steps][n][NZ][NC] (row-major, so A = J[..., :NZ] and B = J[..., NZ:]);
 *   health_dev (unsigned long long[2] or NULL, zeroed by the call): vehicles with a non-finite z or Jacobian entry
 *   in the call / that came within singular_eps (0 = 1e-3) of theta = +-pi/2 at the start of some step.
 * All arrays double, dev. */
typedef struct brov_linearize_desc {
    uint32_t struct_size;       /* = sizeof(brov_linearize_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* z0_dev;
    const void* u_dev;
    long long u_stride_t, u_stride_n;
    void* z_out_dev;
    void* z_traj_dev;
    void* jac_dev;
    void* health_dev;
    double singular_eps;
} brov_linearize_desc;
int brov_linearize(brov_engine_t* e, const brov_linearize_desc* d, void* stream);

/* Closed-loop rollouts: an affine state-feedback law evaluated in the kernel at the start of every integrator step —
 * running an LQR / TVLQR on many vehicles, a robustness Monte-Carlo of a controller over a per-vehicle coefficient
 * table, scoring a controller without storing trajectories.  For vehicle i and step k = 0 .. steps-1, with
 * z_k = [x_k | Z_k] as in brov_linearize (NZ = 30 / 12 / 13 and NU = 8 / 6 / 6 for thruster8 / wrench12 / quat13; Z the
 * allocation-projected lag in [6][3] order):
 *     dz      = z_k - zr_k        Euler-angle models: dz[3..5] -= 2 pi rint(dz[3..5] / 2 pi); quat13: plain difference
 *     u_k     = clamp(ur_k - K_k dz, u_min, u_max)   per channel; a NaN stays NaN (compare-select, not fmin / fmax)
 *     cost   += sum_j q_j dz_j^2 + sum_r r_r (u_k - ur_k)_r^2                       (only with cost_dev)
 *     z_{k+1} = Phi(z_k, u_k)     the step brov_rollout takes (same integrate_step, projected lag)
 * The feedback and the cost are evaluated in the engine's scalar type, every sum in a fixed order with fused
 * multiply-adds, so results are bit-reproducible and independent of the operand layout and of the other vehicles.
 * Operands (engine scalar type) use the rollout's stride addressing, 64-bit:
 *     K  [k*K_stride_t + i*K_stride_n + r*NZ + j]        row-major [NU][NZ], the K numpy builds from a DARE solution
 *     zr [k*z_ref_stride_t + i*z_ref_stride_n + j]
 *     ur [k*u_ref_stride_t + i*u_ref_stride_n + r]
 * so each may be constant and shared (both strides 0), time-varying and shared ([steps][...]), constant per vehicle
 * ([n][...]) or time-varying per vehicle ([steps][n][...]).
 *   u_min / u_max: per-channel bounds (the first NU used; +-INFINITY for none); q[NZ], r[NU]: diagonal cost weights
 *   (unused tails ignored);
 *   z0_dev [n][NZ]; z_out_dev [n][NZ] (required; may alias z0_dev);
 *   traj_dev [steps / stride][n][NZ] or NULL: z after steps stride, 2 stride, ...;
 *   u_traj_dev [steps / stride][n][NU] or NULL: the applied (clamped) input of the step that ends at each snapshot;
 *   cost_dev [n] or NULL: the accumulated cost, added to the incoming values when cost_accumulate (chunked calls add
 *   up bit for bit), else overwritten;
 *   health_dev (unsigned long long[2] or NULL, zeroed by the call): vehicles with a non-finite final z / that came
 *   within singular_eps (0 = 1e-3) of theta = +-pi/2 at the start of some step.
 * Coefficients: the engine's shared set, or its per-vehicle table (brov_set_vehicle_params, pv_n == n).  RK4 / Euler,
 * f64 and f32 engines.  Double-integrator engines and the first-order wrench lag return BROV_EUNSUPPORTED.  BROV_EINVAL:
 * n or steps < 0, dt <= 0, negative strides, NULL K / zr / ur with n * steps > 0, u_min > u_max or a NaN bound, a
 * trajectory without stride >= 1, a table / n mismatch.  n = 0 is a no-op; steps = 0 copies z0 to z_out (and zeroes
 * cost_dev unless cost_accumulate). */
typedef struct brov_closed_loop_desc {
    uint32_t struct_size;       /* = sizeof(brov_closed_loop_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* z0_dev;
    void* z_out_dev;
    const void* K_dev;
    long long K_stride_t, K_stride_n;
    const void* z_ref_dev;
    long long z_ref_stride_t, z_ref_stride_n;
    const void* u_ref_dev;
    long long u_ref_stride_t, u_ref_stride_n;
    double u_min[8], u_max[8];
    double q[30], r[8];
    void* traj_dev;
    void* u_traj_dev;
    long long stride;
    void* cost_dev;
    int32_t cost_accumulate;
    int32_t reserved;
    void* health_dev;
    double singular_eps;
} brov_closed_loop_desc;
int brov_closed_loop(brov_engine_t* e, const brov_closed_loop_desc* d, void* stream);

/* Extended Kalman filters on the Fossen models — state estimation from noisy or partial measurements of the state
 * components (depth, attitude, gyro, DVL, position fixes, each at its own rate), a Monte-Carlo consistency check over
 * many noise realisations, one filter per candidate noise setting scored by likelihood, a fleet of vehicles.
 * For filter i, with z = [x | Z] as in brov_linearize (NX = 12; Z the allocation-projected lag, thruster model only)
 * and k = 0 .. steps-1:
 *   predict   x- = Phi_x(x_k, Z_k, u_k),  Z_{k+1} = Phi_Z(Z_k, u_k)   (the step brov_linearize takes)
 *             P- = A_k P_k A_k^T + diag(q)                          A_k = dx'/dx at (z_k, u_k), NX x NX
 *   update    for j = 0 .. NX-1 with y_k[j] finite, in that order (a NaN marks a component not measured at this
 *             step; +-inf is treated the same way, so a sensor that reports inf for a fault is skipped, not applied):
 *             nu = y_k[j] - x-[j]      (j = 3, 4, 5: wrapped to one turn, nu -= 2 pi rint(nu / 2 pi), as in
 *                                       brov_closed_loop)
 *             s = P-[j][j] + r[j];     g = P-[:, j] (1 / s)    (one division; nu^2 / s below likewise)
 *             x- += g nu;              P- <- (I - g e_j^T) P- (I - g e_j^T)^T + r[j] g g^T      (Joseph form)
 *             loglik -= (nu^2 / s + log s + log 2 pi) / 2;   nis += nu^2 / s;   count += 1
 *   x_{k+1} = x-,  P_{k+1} = P-
 * The measurement model is a selection of state components with diagonal R, so the sequential scalar updates are the
 * joint Kalman update and loglik is the exact Gaussian log-likelihood of the measured components.  y_k measures the
 * state AFTER the step taken with u_k.  The covariance covers x only: Z is a deterministic filter of the known inputs.
 * Only the upper triangle of every P is computed; it is mirrored, so P is exactly symmetric.  Every sum has a fixed
 * order, so results are bit-reproducible and independent of the operand layout and of the other filters.
 * Operands use the rollout's stride addressing, 64-bit:
 *   u [k*u_stride_t + i*u_stride_n + c]   y [k*y_stride_t + i*y_stride_n + j]   (per-filter, shared or constant)
 *   q [i*q_stride_n + j], r [i*r_stride_n + j]   (q_stride_n / r_stride_n = 0: one set shared by every filter)
 *   z0_dev [n][NZ]; P0_dev [n][NX][NX]; z_out_dev [n][NZ] and P_out_dev [n][NX][NX] (required; may alias z0 / P0);
 *   x_traj_dev [steps / stride][n][NX] or NULL: x after steps stride, 2 stride, ...;
 *   P_traj_dev [steps / stride][n][NX][NX] or NULL: P at the same steps;
 *   loglik_dev [n], nis_dev [n] (double), count_dev [n] (int64): all three or none; added to the incoming values when
 *   stats_accumulate (chunked calls add up bit for bit), else overwritten;
 *   health_dev (unsigned long long[2] or NULL, zeroed by the call): filters with a non-finite final z or P / that came
 *   within singular_eps (0 = 1e-3) of theta = +-pi/2 at the start of some step.
 * The engine's shared coefficients, allocation and lag discretisation for dt are used.  fp64 engines, thruster8 and
 * wrench12, RK4 / Euler.  quat13 (the covariance of a unit quaternion is singular), double-integrator engines, the
 * first-order wrench lag, f32 engines and an engine with a per-vehicle coefficient table return BROV_EUNSUPPORTED.
 * BROV_EINVAL: n or steps < 0, dt <= 0, negative strides, q < 0 or r <= 0 (NaN included), NULL required pointers with
 * n * steps > 0, a trajectory without stride >= 1.  n = 0 is a no-op; steps = 0 copies z0 and P0 to the outputs (and
 * zeroes the statistics unless stats_accumulate).  Before the launch the call copies q and r to the host to check
 * them and synchronises `stream` for that copy, so it blocks the calling thread and cannot be captured in a CUDA
 * graph.  All arrays dev. */
typedef struct brov_ekf_desc {
    uint32_t struct_size;       /* = sizeof(brov_ekf_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* z0_dev;
    const void* P0_dev;
    const void* u_dev;
    long long u_stride_t, u_stride_n;
    const void* y_dev;
    long long y_stride_t, y_stride_n;
    const void* q_dev;
    long long q_stride_n;
    const void* r_dev;
    long long r_stride_n;
    void* z_out_dev;
    void* P_out_dev;
    void* x_traj_dev;
    void* P_traj_dev;
    long long stride;
    void* loglik_dev;
    void* nis_dev;
    void* count_dev;
    int32_t stats_accumulate;
    int32_t reserved;
    void* health_dev;
    double singular_eps;
} brov_ekf_desc;
int brov_ekf(brov_engine_t* e, const brov_ekf_desc* d, void* stream);

/* Reverse-mode (adjoint) gradients of batched rollouts — what gradient-based trajectory optimisation, training a policy
 * or a learned model through the simulator, and sensitivity studies need.  With z_{k+1} = Phi(z_k, u_k) the step of
 * brov_linearize (z = [x (NX) | Z (18, thruster model only)], NZ = 30 / 12 / 13, NU = 8 / 6 / 6) and, per vehicle,
 *     L = sum_{k = stride, 2 stride, ... <= steps} <c_k, x_k> + <g_T, z_steps>
 * the call returns gz0 = dL/dz_0 and gu[k] = dL/du_k.  c_k comes from gtraj_dev in the layout of brov_rollout's
 * trajectory, [steps / stride][n][NX] (NULL: no trajectory term); g_T from gzT_dev [n][NZ] (NULL: zero).  The
 * derivative is that of the step brov_linearize differentiates (full sines and cosines in every stage, branch taken:
 * d|x| = sign(x) dx, the clamped cos(theta) and the quaternion fallback are constants; the quaternion renormalised
 * after the step), so gz0 and gu equal the chain lambda_k = A_k^T lambda_{k+1} + c_k, gu_k = B_k^T lambda_{k+1} over
 * brov_linearize's J to rounding, without forming J.  One thread per vehicle runs the forward pass, storing every z_k
 * in the workspace, then the reverse sweep; every sum has a fixed order, so results are bit-reproducible and
 * independent of the input layout and of the other vehicles.
 *   z0_dev [n][NZ]; u_dev with u_stride_t / u_stride_n as in brov_linearize_desc (per-vehicle, shared or constant);
 *   gz0_dev [n][NZ] (required; may alias gzT_dev); gu_dev [steps][n][NU] (required);
 *   z_out_dev [n][NZ] or NULL: z after the last step (the primal of brov_linearize: it agrees with brov_rollout to
 *   rounding, not bit for bit);
 *   workspace_dev: at least brov_rollout_vjp_workspace_bytes(model, n, steps) bytes (n * steps * NZ doubles);
 *   health_dev (unsigned long long[2] or NULL, zeroed by the call): vehicles with a non-finite z, gz0 or gu entry /
 *   that came within singular_eps (0 = 1e-3) of theta = +-pi/2 at the start of some step.
 * Chaining (horizons longer than a workspace allows): split at t1, a multiple of stride when gtraj_dev is used.  The
 * gz0 of the call over [t1, steps], started from z_{t1} = the z_out of a call over [0, t1], is the gzT of the call over
 * [0, t1] (whose gtraj slice ends with c_{t1}).  The chained gradients equal those of one call bit for bit.
 * fp64 engines, Fossen models, RK4 / Euler, the engine's shared coefficients, allocation and lag discretisation for dt.
 * f32 engines, double-integrator engines, the first-order wrench lag and an engine with a per-vehicle coefficient table
 * return BROV_EUNSUPPORTED.  BROV_EINVAL (before any launch): n < 0, steps < 1, dt <= 0, negative input strides, NULL
 * required pointers, gtraj_dev with stride < 1, a workspace smaller than needed.  n = 0 is a no-op.  All arrays double,
 * dev. */
typedef struct brov_rollout_vjp_desc {
    uint32_t struct_size;       /* = sizeof(brov_rollout_vjp_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* z0_dev;
    const void* u_dev;
    long long u_stride_t, u_stride_n;
    const void* gtraj_dev;
    long long stride;
    const void* gzT_dev;
    void* gz0_dev;
    void* gu_dev;
    void* z_out_dev;
    void* workspace_dev;
    size_t workspace_bytes;
    void* health_dev;
    double singular_eps;
} brov_rollout_vjp_desc;
int brov_rollout_vjp(brov_engine_t* e, const brov_rollout_vjp_desc* d, void* stream);
/* workspace of brov_rollout_vjp: n * steps * NZ * sizeof(double) for the Fossen models (0 for other models or n, steps
 * <= 0; SIZE_MAX if the size does not fit in size_t) */
size_t brov_rollout_vjp_workspace_bytes(int model, long long n, long long steps);

/* brov_rollout_vjp plus the gradient of the same L in the kernel coefficients (the BROV_KP_* vector of
 * brov_derive_params) of every vehicle: gkp_dev [BROV_NKP][n] (double, required), gkp[j][i] = dL/dkp_j of vehicle i.
 * Calibration and system identification need it: with phys the physical vector, dL/dphys = gkp^T dkp/dphys (the chain
 * over brov_derive_params), at the cost of one adjoint sweep whatever the number of parameters.  Every stage adds
 * lambda^T df/dkp; the entries of the first-order wrench lag and the pad are 0, the current's are computed whether or
 * not a current is set.  Coefficients: the engine's shared ones, or its per-vehicle table (brov_set_vehicle_params),
 * which must then have n rows (BROV_EINVAL otherwise).  gkp has the table's layout, so the gradient in shared
 * coefficients is the sum of gkp over vehicles.  vjp: every field, refusal and the workspace as for
 * brov_rollout_vjp (vjp.struct_size = sizeof(brov_rollout_vjp_desc)); gx0, gu and z_out are those brov_rollout_vjp
 * returns.  Vehicles with a non-finite gkp entry count in health_dev[0].  Chaining as for brov_rollout_vjp: gz0 and gu
 * are those of one call bit for bit; each call writes the gkp of its own steps, and their sum equals the gkp of one call
 * to rounding. */
typedef struct brov_rollout_vjp_coef_desc {
    uint32_t struct_size;          /* = sizeof(brov_rollout_vjp_coef_desc) */
    int32_t reserved;
    brov_rollout_vjp_desc vjp;
    void* gkp_dev;
} brov_rollout_vjp_coef_desc;
int brov_rollout_vjp_coef(brov_engine_t* e, const brov_rollout_vjp_coef_desc* d, void* stream);

/* Reverse-mode gradients of closed-loop rollouts (brov_closed_loop) — tuning a feedback gain over a fleet of perturbed
 * vehicles, optimising the feedforward reference of a tracking controller, training a policy with feedback in the
 * loop.  In the notation of brov_closed_loop, per vehicle and step k:
 *     dz_k = wrap(z_k - zr_k)     v_k = ur_k - K_k dz_k     u_k = clamp(v_k, u_min, u_max)     z_{k+1} = Phi(z_k, u_k)
 *     cost = sum_k sum_j q_j dz_kj^2 + sum_r r_r (u_k - ur_k)_r^2
 *     L    = sum_{k = stride, 2 stride, ... <= steps} <c_k, z_k> + <g_T, z_steps> + g_c cost
 * the call returns gz0 = dL/dz_0 and, each when its pointer is not NULL, dL/dK, dL/dzr and dL/dur in the layout of the
 * operand as passed (same strides): an element read by several steps or vehicles (a zero stride) receives the sum of
 * their contributions, the gradient of an operand of that shape.  Per step and vehicle the cotangents are
 *     gv = m . (B_k^T lambda_{k+1} + 2 g_c r . (u_k - ur_k))    (m: 0 on a clamped channel, else 1; a NaN is not clamped)
 *     dL/dK_k = -gv dz_k^T     dL/dzr_k = -gdz     dL/dur_k = gv - 2 g_c r . (u_k - ur_k)
 *     gdz = -K_k^T gv + 2 g_c q . dz_k                 lambda_k = A_k^T lambda_{k+1} + gdz + c_k
 * with A, B the step's Jacobians as brov_rollout_vjp differentiates them and d wrap = 1.  The primal is
 * brov_linearize's step, so z_out agrees with brov_closed_loop to rounding, not bit for bit.  One thread per vehicle
 * runs the forward pass (z_k to the workspace) and the reverse sweep (u_k recomputed from z_k, never stored); the
 * operand gradients are then summed by separate kernels in a fixed order, without floating-point atomics.  Results are
 * bit-reproducible; gz0 and the gradients of per-vehicle layouts do not depend on the other vehicles or on which
 * layout holds equal values.
 *   integrator, n, steps, dt, z0_dev, K / z_ref / u_ref with their strides, u_min / u_max, q, r: as brov_closed_loop_desc;
 *   gtraj_dev [steps / stride][n][NZ] or NULL: c_k on the full z (closed_loop's traj layout); gzT_dev [n][NZ] or NULL;
 *   gcost_dev [n] or NULL: g_c per vehicle (NULL: no cost term);
 *   gz0_dev [n][NZ] (required; may alias gzT_dev); gK_dev, gz_ref_dev, gu_ref_dev or NULL; z_out_dev [n][NZ] or NULL;
 *   workspace_dev: brov_closed_loop_vjp_workspace_bytes(model, n, steps) bytes always suffice; fewer operand
 *   gradients need less: n * steps doubles times (NZ, + NU with gK, + NZ with gz_ref, + NU with gu_ref), plus n * E
 *   doubles when an operand of E elements whose gradient is requested has both strides 0;
 *   health_dev (unsigned long long[2] or NULL, zeroed by the call): vehicles with a non-finite z, gz0 or per-step
 *   operand-gradient entry (dL/dur_k, dL/dzr_k and, with gK_dev, dL/dK_k = -gv dz_k^T) / that came within singular_eps
 *   (0 = 1e-3) of theta = +-pi/2 at the start of some step.
 * Chaining: split at t1 as for brov_rollout_vjp (gtraj, K, z_ref and u_ref sliced at t1 when time-varying).  gz0 and the
 * time-sliced gradients (shared and per-vehicle time-varying layouts) equal those of one call bit for bit; each call
 * writes the sums of a constant layout over its own steps, and these add up to the one-call result to rounding.
 * Coefficients: the engine's shared set, or its per-vehicle table (n rows).  fp64 engines, Fossen models, RK4 / Euler.
 * f32 engines, double-integrator engines and the first-order wrench lag return BROV_EUNSUPPORTED.  BROV_EINVAL (before
 * any launch): every input brov_closed_loop refuses, steps < 1, gtraj_dev with stride < 1, NULL gz0, a requested
 * operand gradient whose strides make distinct (step, vehicle) pairs overlap, a workspace smaller than needed, a
 * table / n mismatch.  n = 0 is a no-op.  All arrays double, dev. */
typedef struct brov_closed_loop_vjp_desc {
    uint32_t struct_size;       /* = sizeof(brov_closed_loop_vjp_desc) */
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* z0_dev;
    const void* K_dev;
    long long K_stride_t, K_stride_n;
    const void* z_ref_dev;
    long long z_ref_stride_t, z_ref_stride_n;
    const void* u_ref_dev;
    long long u_ref_stride_t, u_ref_stride_n;
    double u_min[8], u_max[8];
    double q[30], r[8];
    const void* gtraj_dev;
    long long stride;
    const void* gzT_dev;
    const void* gcost_dev;
    void* gz0_dev;
    void* gK_dev;
    void* gz_ref_dev;
    void* gu_ref_dev;
    void* z_out_dev;
    void* workspace_dev;
    size_t workspace_bytes;
    void* health_dev;
    double singular_eps;
} brov_closed_loop_vjp_desc;
int brov_closed_loop_vjp(brov_engine_t* e, const brov_closed_loop_vjp_desc* d, void* stream);
/* workspace of brov_closed_loop_vjp with every operand gradient requested: n * (steps * (2 NZ + 2 NU) + NU * NZ)
 * doubles for the Fossen models (0 for other models or n, steps <= 0; SIZE_MAX if the size does not fit in size_t) */
size_t brov_closed_loop_vjp_workspace_bytes(int model, long long n, long long steps);

/* Reduced 9-state RHS — `bluerov_compute(t, x_, u_)` (fossen/bluerov_torch.py:20-67, constants fossen/parameters.py).
 * x [B][9], u [B][4], out [B][9]. */
int brov_reduced9_rhs(int dtype, const void* x_dev, const void* u_dev, void* out_dev, long long B, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Koopman EDMDc comparison model — scoring and simulation of a FITTED model (Koopman/koopmanEDMDc.py; the fit itself,
 * k-means centres + a ridge normal-equation solve, stays host work as in the reference).  All arithmetic float64.
 *   phi(x) = [x, exp(-gamma (|x|^2 + |c_j|^2 - 2 x.c_j))_j], d = n + k          _lift / _rbf_mat  :41-49, 221-238
 * create: centers [k][n], A [d][d], B [d][r] are HOST arrays (row-major double), copied to the device.
 * Supported (n, r): (12, 8), (12, 6), (13, 6); d limited by shared memory (d = 512 fits). */
typedef struct brov_koopman brov_koopman_t;
int brov_koopman_create(int device, int n, int r, int k, double gamma, const double* centers, const double* A,
                        const double* B, brov_koopman_t** out);
void brov_koopman_destroy(brov_koopman_t* h);
/* Z[rows][d] = phi(X[rows][n])                                                    _lift :221-238 */
int brov_koopman_lift(brov_koopman_t* h, const double* X_dev, long long rows, double* Z_dev, void* stream);
/* Sum over windows w in [0, n_windows) of |x_hat_w - X[w+H]|^2 with x_hat_w = first n coordinates of the lifted state
 * propagated H steps from phi(X[w]) under U[w..w+H-1] — `multistep_rmse(X, U, H)` :172-200 with n_windows = rows - H
 * (rmse = sqrt(se / (n_windows n))), and `evaluate(X, U)` :157-170 for H = 1.  se_out_dev: double[1], dev. */
int brov_koopman_multistep_se(brov_koopman_t* h, const double* X_dev, const double* U_dev, long long rows,
                              long long n_windows, int H, double* se_out_dev, void* stream);
/* The same for up to BROV_MAX_H horizons in one call (horizons: host array, strictly ascending): the lift phi(x_k) is
 * evaluated once per window and pushed through the decoder rows of every horizon; horizon h scores windows
 * 0 .. rows - H_h - 1.  se_out_dev: double[n_horizons], dev. */
int brov_koopman_multistep_se_multi(brov_koopman_t* h, const double* X_dev, const double* U_dev, long long rows,
                                    int n_horizons, const int* horizons, double* se_out_dev, void* stream);
/* `simulate(x0, U_seq)` :202-216 for nb trajectories at once: X0 [nb][n]; U time-major [T][nb][r] (u_shared = 0) or
 * [T][r] (u_shared = 1); out [T][nb][n] = predicted states after steps 1..T (row 0 of the reference's array is x0). */
int brov_koopman_simulate(brov_koopman_t* h, const double* X0_dev, const double* U_dev, long long T, long long nb,
                          int u_shared, double* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * PINc comparison model — inference of the reference's residual network x_{k+1} = x_k + f([x_k, u_k, dt]) on the
 * 9-state [x y z cos(psi) sin(psi) u v w r] with inputs [X Y Z Mz] from the thruster map (training/
 * train_tank_brov2_rk4.py:553-840).  Network arithmetic is float32 (as torch runs it), the thruster map float64.
 * Weights: the tensors of PINcNet.state_dict() (14 -> 64 -> 64 -> 64 -> 64 -> 9; Linear / AdaptiveSoftplus / LayerNorm
 * per hidden layer), HOST float arrays in torch's layouts: W[l] is [out][in] row-major. */
typedef struct brov_pinc brov_pinc_t;
typedef struct brov_pinc_weights {
    uint32_t struct_size;
    int32_t n_hidden_layers;    /* 4 */
    int32_t hidden;             /* 64 */
    int32_t reserved;
    const float* W[5];          /* net.0 / net.3 / net.6 / net.9 / net.12 .weight */
    const float* b[5];          /* ... .bias */
    float beta[4];              /* net.1 / net.4 / net.7 / net.10 .beta */
    const float* ln_w[4];       /* net.2 / net.5 / net.8 / net.11 .weight */
    const float* ln_b[4];       /* ... .bias */
} brov_pinc_weights;
int brov_pinc_create(int device, const brov_pinc_weights* w, brov_pinc_t** out);
void brov_pinc_destroy(brov_pinc_t* h);
/* Thruster map constants for the sampling time the rollouts run at: (Ad, Bd) from brov_lag_discretize(dt), alloc
 * [6][8] from brov_default_allocation (thrusters_to_body_wrenches, :553-562). */
int brov_pinc_set_thruster_map(brov_pinc_t* h, double dt, const double* Ad, const double* Bd, const double* alloc);
/* PINcNet.forward (:627-673): z [n][14] = [x9, u4, dt] float -> x9_next [n][9] float. */
int brov_pinc_forward(brov_pinc_t* h, const float* z_dev, float* out_dev, long long n, void* stream);
/* simulate_pinc (:789-812) for n windows at once.  x0 [n][12] double (12-state rows), inputs as in brov_rollout
 * (8 thruster voltages, double), lag_in [n][8][3] double or NULL = zeros; lag_out [n][4][3] double or NULL: the
 * allocation-projected lag of the X, Y, Z, Mz rows; traj [steps/stride][n][12] double or NULL: 12-state projection
 * (state9_to_12: phi = theta = p = q = 0, psi = atan2) after steps stride, 2 stride, ...; x9T [n][9] float or NULL. */
typedef struct brov_pinc_rollout_desc {
    uint32_t struct_size;
    int32_t reserved;
    long long n;
    long long steps;
    const void* x0_dev;
    const void* u_dev;
    long long u_stride_t, u_stride_n;
    const void* lag_in_dev;
    void* lag_out_dev;
    void* traj_dev;
    long long stride;
    void* x9T_dev;
} brov_pinc_rollout_desc;
int brov_pinc_rollout(brov_pinc_t* h, const brov_pinc_rollout_desc* d, void* stream);
/* multistep_rmse_endpoint_pinc (:815-840): as brov_multistep_se on X [rows][12], U [rows][8] (double).  carry_steps
 * = 0: every window starts from zero lag; > 0 (one horizon): the reference's literal behaviour — one thruster-map
 * object scores all windows in order — reproduced by replaying the last carry_steps lag steps of that history
 * (brov_se_carry_steps(thruster engine, dt, BROV_EULER)).  se_out_dev: double[BROV_MAX_H], dev. */
typedef struct brov_pinc_se_desc {
    uint32_t struct_size;
    int32_t n_horizons;
    int32_t horizons[BROV_MAX_H];
    long long rows;
    long long n_windows;
    const void* X_dev;
    const void* U_dev;
    double* se_out_dev;
    int32_t carry_steps;
    int32_t reserved;
    long long window0;
    long long row0;
    const void* carry_lag0_dev;  /* [8][3] double: lag state of the thruster-map object before window 0, or NULL = zeros */
} brov_pinc_se_desc;
int brov_pinc_multistep_se(brov_pinc_t* h, const brov_pinc_se_desc* d, void* stream);

/* Host-buffer rollout: the same operation as brov_rollout with every array in HOST memory (pinned memory gives
 * asynchronous copies).  The engine streams the inputs to the device in time chunks on a copy stream, double
 * buffered against the rollout kernels, and copies snapshots and final state back; it returns after everything has
 * landed in the host arrays.  u_host is time-major [steps][n][NU] (u_shared = 0) or [steps][NU] (u_shared = 1).
 * Chunks carry the allocation-projected lag on the device; per-thruster states (lag_out_repr = BROV_LAG_THRUSTER) are
 * rebuilt from the chunks that cover the last brov_se_carry_steps steps. */
typedef struct brov_rollout_host_desc {
    uint32_t struct_size;
    int32_t integrator;
    long long n;
    long long steps;
    double dt;
    const void* x0_host;        /* [n][NX] */
    void* xT_host;              /* [n][NX] */
    const void* u_host;
    int32_t u_shared;
    int32_t reserved;
    const void* lag_in_host;    /* or NULL */
    void* lag_out_host;         /* or NULL */
    void* traj_host;            /* [steps/stride][n][NX] or NULL */
    long long stride;
    long long chunk_steps;      /* 0 = choose (about 256 MiB of inputs per chunk) */
    int32_t lag_in_repr;        /* BROV_LAG_*: layout of lag_in_host / lag_out_host (thruster model only) */
    int32_t lag_out_repr;
    /* generated inputs (gen.enable): u_host is ignored, nothing but x0 / lag / the AR(1) state crosses PCIe;
     * gen.state_in_dev / state_out_dev are HOST pointers here ([n][NU] or NULL) */
    brov_input_gen gen;
    unsigned long long* health_host;   /* [2] or NULL: non-finite / near-singular vehicle counts of the whole call */
    double singular_eps;               /* 0 = 1e-3 */
} brov_rollout_host_desc;
int brov_rollout_host(brov_engine_t* e, const brov_rollout_host_desc* d);

/* Pinned host memory helpers for brov_rollout_host callers without their own allocator. */
int brov_host_alloc(size_t bytes, void** out);
int brov_host_free(void* p);

/* FMA-chain microbenchmark on `device`: the FP32 / FP64 pipe peak used as roofline denominator. */
int brov_fma_peak(int dtype, int device, int iters, double* tflops_out, double* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* BROV_H */
