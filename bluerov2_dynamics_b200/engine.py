"""Host side of the B200 engine: torch provides device memory and streams, libbrov.so (C ABI) does the work.

`Engine` is the batched counterpart of the reference's model objects: where the reference evaluates one vehicle per
Python call (`rov.dynamics`, `simulate_physics`, `multistep_rmse_endpoint_physics`), an Engine call covers N
vehicles / windows with one kernel launch.  Array conventions follow the reference: a state is a row
`[x y z phi theta psi u v w p q r]` (or the 13-state quaternion row), an input row is 8 thruster voltages or a
6-component body wrench.
"""
from __future__ import annotations

import ctypes as C
from contextlib import contextmanager, nullcontext as _nullcontext
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib as L

MODELS = {"thruster8": L.THRUSTER8_LAG3, "wrench12": L.WRENCH_EULER12, "quat13": L.WRENCH_QUAT13,
          # double-integrator comparison model: 12-state with 8 thruster / 6 wrench inputs, 13-state quaternion
          "di12_u8": L.DI_EULER12_U8, "di12_u6": L.DI_EULER12_U6, "diq13_u6": L.DI_QUAT13_U6}
_NX13 = ("quat13", "diq13_u6")
_NU8 = ("thruster8", "di12_u8")
DTYPES = {"f64": (L.F64, torch.float64, np.float64), "f32": (L.F32, torch.float32, np.float32)}
INTEGRATORS = {"rk4": L.RK4, "euler": L.EULER}
SWEEP_WORKSPACE_CAP = 256 << 20   # bytes of sweep workspace per launch (Engine.multistep_se_sweep splits P to fit)


def default_physical(rho: float = 1000.0) -> np.ndarray:
    """Scalar attributes of the reference classes as one vector (layout: include/brov.h BROV_PH_*)."""
    ph = np.zeros(L.NPHYS)
    L.check(L.lib.brov_default_physical(float(rho), L.dptr(ph)))
    return ph


def derive_params(phys: np.ndarray) -> np.ndarray:
    """Physical vector(s) [..., NPHYS] -> kernel coefficient vector(s) [..., NKP] (float64, host)."""
    phys = np.ascontiguousarray(phys, dtype=np.float64)
    flat = phys.reshape(-1, L.NPHYS)
    out = np.zeros((flat.shape[0], L.NKP))
    for i in range(flat.shape[0]):
        L.check(L.lib.brov_derive_params(L.dptr(flat[i]), L.dptr(out[i])))
    return out.reshape(phys.shape[:-1] + (L.NKP,))


def with_minv(phys: np.ndarray) -> np.ndarray:
    """Copy of physical vector(s) [..., NPHYS] whose diag(Minv) entries are rebuilt from m, the inertias and the added
    masses, as the reference's __init__ computes them: 1/(m - X_udot), ..., 1/(Iz - N_rdot).  The kernels use the Minv
    they are given (the reference freezes it at construction, SURVEY trap T5), so a candidate table that perturbs the
    masses must pass through this to describe the vehicle it means."""
    ph = np.array(phys, dtype=np.float64)
    m = ph[..., L.PH_M:L.PH_M + 1]
    ph[..., L.PH_MINV:L.PH_MINV + 3] = 1.0 / (m - ph[..., L.PH_ADDED:L.PH_ADDED + 3])
    ph[..., L.PH_MINV + 3:L.PH_MINV + 6] = 1.0 / (ph[..., L.PH_I:L.PH_I + 3] - ph[..., L.PH_ADDED + 3:L.PH_ADDED + 6])
    return ph


# kernel coefficient vector layout (include/brov.h, csrc/brov_device.cuh KP_*)
KP_MINV, KP_A, KP_DA, KP_DB, KP_DL, KP_DQ, KP_WMB, KP_XBB, KP_CUR = 0, 6, 9, 12, 15, 21, 27, 28, 31


def derive_params_torch(phys: torch.Tensor, rebuild_minv: bool = True) -> torch.Tensor:
    """Differentiable torch twin of derive_params(with_minv(phys)) (of derive_params(phys) without rebuild_minv):
    physical vector(s) [..., NPHYS] -> kernel coefficients [..., NKP], same dtype and device, so that dL/dphys follows
    from a coefficient gradient (Engine.rollout_diff(kp=...), Engine.rollout_vjp(coef=True)) by autograd.  Its
    Jacobian is coefficient_directions.  The first-order wrench lag entry (1/T_lag1, 0 without a lag) carries no
    gradient."""
    ph = phys
    m = ph[..., L.PH_M:L.PH_M + 1]
    a = m - ph[..., L.PH_ADDED:L.PH_ADDED + 3]
    b = ph[..., L.PH_I:L.PH_I + 3] - ph[..., L.PH_ADDED + 3:L.PH_ADDED + 6]
    minv = torch.cat([1.0 / a, 1.0 / b], dim=-1) if rebuild_minv else ph[..., L.PH_MINV:L.PH_MINV + 6]
    a0, a1, a2 = a.unbind(-1)
    b0, b1, b2 = b.unbind(-1)
    B = ph[..., L.PH_B:L.PH_B + 1]
    tl = ph[..., L.PH_TLAG1:L.PH_TLAG1 + 1].detach()
    ilag = torch.where(tl > 0.0, 1.0 / torch.where(tl > 0.0, tl, torch.ones_like(tl)), torch.zeros_like(tl))
    return torch.cat([minv, a, torch.stack([a2 - a1, a0 - a2, a1 - a0], dim=-1),
                      torch.stack([b2 - b1, b0 - b2, b1 - b0], dim=-1),
                      -ph[..., L.PH_LIN:L.PH_LIN + 6], -ph[..., L.PH_QUAD:L.PH_QUAD + 6],
                      ph[..., L.PH_W:L.PH_W + 1] - B, ph[..., L.PH_XB:L.PH_XB + 3] * B,
                      ph[..., L.PH_CURRENT:L.PH_CURRENT + 3], ilag, torch.zeros_like(ilag)], dim=-1)

# names of the physical vector's entries: the reference's attribute names (fossen/BlueROV2.py:81-150); the ocean
# current is `current_speed` split into its NED components, diag(Minv) is named after the velocity it scales
_AXES = ("u", "v", "w", "p", "q", "r")
PHYS_NAMES = (["m", "W", "B", "xb", "yb", "zb", "Ix", "Iy", "Iz"]
              + ["Xu_dot", "Yv_dot", "Zw_dot", "Kp_dot", "Mq_dot", "Nr_dot"]
              + ["Xu", "Yv", "Zw", "Kp", "Mq", "Nr"]
              + ["Xu_abs", "Yv_abs", "Zw_abs", "Kp_abs", "Mq_abs", "Nr_abs"]
              + [f"Minv_{a}" for a in _AXES]
              + ["current_n", "current_e", "current_d", "T_lag1"])
PARAM_GROUPS = {"added": list(range(L.PH_ADDED, L.PH_ADDED + 6)), "lin": list(range(L.PH_LIN, L.PH_LIN + 6)),
                "quad": list(range(L.PH_QUAD, L.PH_QUAD + 6)),
                "current": list(range(L.PH_CURRENT, L.PH_CURRENT + 3))}


def parameter_indices(params) -> list:
    """Physical-vector indices of a parameter selection: PH_* indices, attribute names (PHYS_NAMES) or the groups
    "added", "lin", "quad", "current", in any mix.  The first-order wrench lag (T_lag1) is not a parameter."""
    if isinstance(params, (str, int, np.integer)):
        params = [params]
    idx = []
    for q in params:
        if isinstance(q, (int, np.integer)):
            if not 0 <= int(q) < L.NPHYS:
                raise ValueError(f"parameter index {q} out of range")
            idx.append(int(q))
        elif q in PARAM_GROUPS:
            idx.extend(PARAM_GROUPS[q])
        elif q in PHYS_NAMES:
            idx.append(PHYS_NAMES.index(q))
        else:
            raise ValueError(f"unknown parameter {q!r}: use a PH_* index, one of {PHYS_NAMES[:-1]} or a group "
                             f"{list(PARAM_GROUPS)}")
    if L.PH_TLAG1 in idx:
        raise ValueError("T_lag1 (the first-order wrench lag) is not supported as a parameter")
    if len(set(idx)) != len(idx):
        raise ValueError("a parameter is selected twice")
    if not 1 <= len(idx) <= L.NKP:
        raise ValueError(f"select 1..{L.NKP} parameters")
    return idx


def coefficient_directions(phys: np.ndarray, params, rebuild_minv: bool = True) -> np.ndarray:
    """Analytic Jacobian [p, NKP] of the kernel coefficients in the selected physical parameters at `phys`: row j is
    d derive_params(with_minv(phys)) / d phys[params[j]] (without with_minv if rebuild_minv is False).
    With rebuild_minv, diag(Minv) follows m, the inertias and the added masses as the reference's __init__ computes it,
    and the Minv entries cannot be parameters; without it they are parameters of their own (the reference freezes
    Minv at construction, SURVEY trap T5)."""
    ph = np.asarray(phys, dtype=np.float64).reshape(L.NPHYS)
    idx = parameter_indices(params)
    if rebuild_minv and any(L.PH_MINV <= i < L.PH_MINV + 6 for i in idx):
        raise ValueError("Minv entries follow the masses with rebuild_minv=True: select them with rebuild_minv=False")
    add = ph[L.PH_ADDED:L.PH_ADDED + 6]
    a = ph[L.PH_M] - add[:3]                       # m - X_udot, ...
    b = ph[L.PH_I:L.PH_I + 3] - add[3:]            # Ix - K_pdot, ...
    D = np.zeros((len(idx), L.NKP))
    for r, i in enumerate(idx):
        row, da, db = D[r], np.zeros(3), np.zeros(3)
        if i == L.PH_M:
            da[:] = 1.0
        elif i == L.PH_W:
            row[KP_WMB] = 1.0
        elif i == L.PH_B:
            row[KP_WMB] = -1.0
            row[KP_XBB:KP_XBB + 3] = ph[L.PH_XB:L.PH_XB + 3]
        elif L.PH_XB <= i < L.PH_XB + 3:
            row[KP_XBB + i - L.PH_XB] = ph[L.PH_B]
        elif L.PH_I <= i < L.PH_I + 3:
            db[i - L.PH_I] = 1.0
        elif L.PH_ADDED <= i < L.PH_ADDED + 3:
            da[i - L.PH_ADDED] = -1.0
        elif L.PH_ADDED + 3 <= i < L.PH_ADDED + 6:
            db[i - L.PH_ADDED - 3] = -1.0
        elif L.PH_LIN <= i < L.PH_LIN + 6:
            row[KP_DL + i - L.PH_LIN] = -1.0
        elif L.PH_QUAD <= i < L.PH_QUAD + 6:
            row[KP_DQ + i - L.PH_QUAD] = -1.0
        elif L.PH_MINV <= i < L.PH_MINV + 6:
            row[KP_MINV + i - L.PH_MINV] = 1.0
        else:                                      # ocean current
            row[KP_CUR + i - L.PH_CURRENT] = 1.0
        row[KP_A:KP_A + 3] += da
        row[KP_DA:KP_DA + 3] += [da[2] - da[1], da[0] - da[2], da[1] - da[0]]
        row[KP_DB:KP_DB + 3] += [db[2] - db[1], db[0] - db[2], db[1] - db[0]]
        if rebuild_minv:
            row[KP_MINV:KP_MINV + 3] -= da / a ** 2
            row[KP_MINV + 3:KP_MINV + 6] -= db / b ** 2
    return D


@dataclass
class GradResult:
    """Endpoint error and its exact derivatives in the selected parameters (Engine.multistep_se_grad)."""
    se: torch.Tensor                 # [nH] float64: sum over windows of |r_w|^2 per horizon
    grad: torch.Tensor               # [nH, p]: d se / d theta
    gn: torch.Tensor                 # [nH, p, p]: Gauss-Newton matrix sum_w J_w^T J_w (exactly symmetric)
    counts: list                     # windows per horizon
    names: list                      # parameter names (PHYS_NAMES)
    index: list                      # their physical-vector indices


@dataclass
class LinearizeResult:
    """Exact Jacobians of every step along N trajectories (Engine.linearize), in projected lag coordinates."""
    A: torch.Tensor                  # [T, N, NZ, NZ] dz_{k+1} / dz_k   (view of one J [T, N, NZ, NZ+NU])
    B: torch.Tensor                  # [T, N, NZ, NU] dz_{k+1} / du_k   (view of the same J)
    z: torch.Tensor                  # [N, NZ] z after the last step
    z_traj: Optional[torch.Tensor]   # [T, N, NZ] z after every step, or None
    health: Optional[torch.Tensor]   # int64 [2]: vehicles with a non-finite result / near theta = +-pi/2, or None


@dataclass
class ClosedLoopResult:
    """Closed-loop rollout of N vehicles under affine state feedback (Engine.closed_loop), projected lag coordinates."""
    z: torch.Tensor                  # [N, NZ] z after the last step
    z_traj: Optional[torch.Tensor]   # [S, N, NZ] z after steps stride, 2 stride, ..., or None
    u_traj: Optional[torch.Tensor]   # [S, N, NU] the applied (clamped) input of the step ending at each snapshot, or None
    cost: Optional[torch.Tensor]     # [N] accumulated stage cost (engine scalar type), or None
    health: Optional[torch.Tensor]   # int64 [2]: vehicles with a non-finite final z / near theta = +-pi/2, or None


@dataclass
class EkfResult:
    """N extended Kalman filters run over one measurement series each (Engine.ekf), projected lag coordinates."""
    z: torch.Tensor                  # [N, NZ] the estimate z = [x | Z] after the last step
    P: torch.Tensor                  # [N, NX, NX] its covariance (exactly symmetric)
    x_traj: Optional[torch.Tensor]   # [S, N, NX] the state estimate after steps stride, 2 stride, ..., or None
    P_traj: Optional[torch.Tensor]   # [S, N, NX, NX] the covariance at the same steps (want_cov), or None
    loglik: torch.Tensor             # [N] float64 log-likelihood of the measurements
    nis: torch.Tensor                # [N] float64 sum of the normalised innovations squared
    count: torch.Tensor              # [N] int64 number of scalar measurements used
    health: Optional[torch.Tensor]   # int64 [2]: filters with a non-finite z or P / near theta = +-pi/2, or None


@dataclass
class VjpResult:
    """Reverse-mode gradients of N rollouts (Engine.rollout_vjp) for L = sum_k <c_k, x_k> + <g_T, z_T>."""
    gx0: torch.Tensor                # [N, NX] dL/dx_0
    glag0: Optional[torch.Tensor]    # dL/dlag_0 in the representation of lag0 ([N, 24] or [N, 18]), None for wrench models
    gU: torch.Tensor                 # [T, N, NU] dL/du_k (always per vehicle)
    z: torch.Tensor                  # [N, NZ] z after the last step (the primal of linearize, projected lag)
    health: Optional[torch.Tensor]   # int64 [2]: vehicles with a non-finite z or gradient / near theta = +-pi/2, or None
    gkp: Optional[torch.Tensor] = None   # [N, NKP] dL/dkp of each vehicle's coefficients (coef=True), or None


@dataclass
class ClosedLoopVjpResult:
    """Reverse-mode gradients of N closed-loop rollouts (Engine.closed_loop_vjp), each operand gradient in the shape of
    the operand passed (a layout with a shared dimension gets the sum over it)."""
    gx0: torch.Tensor                # [N, NX] dL/dx_0
    glag0: Optional[torch.Tensor]    # dL/dlag_0 in the representation of lag0 ([N, 24] or [N, 18]), None for wrench models
    gK: Optional[torch.Tensor]       # dL/dK, or None when not wanted
    gz_ref: Optional[torch.Tensor]   # dL/dz_ref, or None when not wanted
    gu_ref: Optional[torch.Tensor]   # dL/du_ref, or None when not wanted
    z: torch.Tensor                  # [N, NZ] z after the last step (the primal of linearize, projected lag)
    health: Optional[torch.Tensor]   # int64 [2]: vehicles with a non-finite z or gradient / near theta = +-pi/2, or None


_CL_LAYOUTS = ("const_shared", "shared", "const", "tnc")


def default_allocation():
    """(alloc [6,8], r [8,3], dir [8,3]) from the reference's thruster geometry formula."""
    a, r, d = np.zeros((6, 8)), np.zeros((8, 3)), np.zeros((8, 3))
    L.check(L.lib.brov_default_allocation(L.dptr(a), L.dptr(r), L.dptr(d)))
    return a, r, d


def lag_discretize(dt: float):
    """(Ad [3,3], Bd [3]): zero-order hold of the 3rd-order thruster lag at sampling time dt."""
    Ad, Bd = np.zeros((3, 3)), np.zeros(3)
    L.check(L.lib.brov_lag_discretize(float(dt), L.dptr(Ad), L.dptr(Bd)))
    return Ad, Bd


@dataclass
class RolloutResult:
    xT: torch.Tensor                 # [N, NX]
    lag: Optional[torch.Tensor]      # [N, NLAG] or None
    traj: Optional[torch.Tensor]     # [S, N, NX] or None
    gen_state: Optional[torch.Tensor] = None     # [N, NU] AR(1) state of the generated command signal after the call
    health: Optional[torch.Tensor] = None        # int64 [2]: vehicles with a non-finite final state / near theta = +-pi/2
    min_abs_cos: Optional[torch.Tensor] = None   # [N] running minimum of |cos theta|


@dataclass
class InputGenerator:
    """The reference's smooth random command signal (training/train_sim_brov2_koopmanEDMDc.py:161-164,180)
        u_k = scale * s_k,   s_k = clip(rho s_{k-1} + sigma N(0,1), -clip, clip),   s_{-1} = 0
    generated INSIDE the rollout kernels from the counter-based Philox4x32-10 stream keyed on (seed, vehicle0 + i,
    step0 + k): no input array in HBM, the same numbers whatever the chunking / slicing / sharding."""
    seed: int = 0
    rho: float = 0.98
    sigma: float = 0.02
    clip: float = 1.0
    scale: Optional[Sequence[float]] = None      # per input channel, default 1
    vehicle0: int = 0                            # global index of the engine's vehicle 0 (rank offset of a shard)

    def fill(self, g: "L.InputGen", nu: int, state_in=None, state_out=None) -> None:
        g.enable = 1
        g.seed = int(self.seed) & 0xFFFFFFFFFFFFFFFF
        g.vehicle0 = int(self.vehicle0)
        g.rho, g.sigma, g.clip = float(self.rho), float(self.sigma), float(self.clip)
        sc = [1.0] * nu if self.scale is None else [float(v) for v in self.scale]
        if len(sc) != nu:
            raise ValueError(f"scale must have {nu} entries")
        for j in range(8):
            g.scale[j] = sc[j] if j < nu else 0.0
        g.state_in_dev = state_in
        g.state_out_dev = state_out


class Engine:
    def __init__(self, model: str = "thruster8", dtype: str = "f64", device: Optional[int] = None,
                 rho: float = 1000.0, current: Optional[Sequence[float]] = None):
        if model not in MODELS:
            raise ValueError(f"model must be one of {list(MODELS)}")
        if dtype not in DTYPES:
            raise ValueError(f"dtype must be one of {list(DTYPES)}")
        if not torch.cuda.is_available():
            raise RuntimeError("bluerov2_dynamics_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.model, self.dtype = model, dtype
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self._code, self.tdtype, self.ndtype = DTYPES[dtype]
        self.nx = 13 if model in _NX13 else 12
        self.nu = 8 if model in _NU8 else 6
        self.is_di = model.startswith("di")
        self._lag1 = False
        h = C.c_void_p()
        L.check(L.lib.brov_create(MODELS[model], self._code, self.device_index, C.byref(h)))
        self._h = h
        self._pv = None
        self._pv_current = False
        self._ws = None
        self._alloc = None if self.is_di else default_allocation()[0]   # last allocation pushed to the library
        self.phys = default_physical(rho)
        if current is not None:
            self.phys[L.PH_CURRENT:L.PH_CURRENT + 3] = np.asarray(current, float).reshape(3)
        self.set_physical(self.phys)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "lib", None) is not None:   # module globals may be gone at shutdown
            L.lib.brov_destroy(h)
            self._h = None

    # ------------------------------------------------------------------ constants
    @property
    def nlag(self) -> int:
        return 24 if self.model == "thruster8" else (6 if self._lag1 else 0)

    def set_physical(self, phys: np.ndarray) -> None:
        """Constants shared by all vehicles, from a physical vector (BROV_PH_* layout)."""
        self.phys = np.array(phys, dtype=np.float64).reshape(L.NPHYS)
        kp = derive_params(self.phys)
        L.check(L.lib.brov_set_params(self._h, L.dptr(kp)))

    def set_vehicle_physical(self, phys_table: Optional[np.ndarray]) -> None:
        """Per-vehicle (Monte-Carlo) constants: phys_table [N, NPHYS] or None to clear."""
        if phys_table is None:
            self._pv = None
            L.check(L.lib.brov_set_vehicle_params(self._h, None, 0, 0))
            return
        kp = derive_params(np.asarray(phys_table, float))          # [N, NKP]
        soa = torch.from_numpy(np.ascontiguousarray(kp.T)).to(self.device, self.tdtype).contiguous()  # [NKP, N]
        self._pv = soa
        any_current = bool(np.any(np.asarray(phys_table, float)[..., L.PH_CURRENT:L.PH_CURRENT + 3] != 0.0))
        self._pv_current = any_current
        L.check(L.lib.brov_set_vehicle_params(self._h, soa.data_ptr(), soa.shape[1], int(any_current)))

    @contextmanager
    def _coefficients(self, kp: torch.Tensor):
        """Runs the body with the kernel coefficients kp (float64 [NKP]: shared, [N, NKP]: a per-vehicle table) in
        place of the engine's own, which are restored afterwards, also when the body raises."""
        k = kp.detach()
        try:
            if k.dim() == 1:
                L.check(L.lib.brov_set_vehicle_params(self._h, None, 0, 0))
                L.check(L.lib.brov_set_params(self._h, L.dptr(np.ascontiguousarray(k.cpu().numpy()))))
            else:
                soa = k.t().contiguous()
                cur = bool((k[:, KP_CUR:KP_CUR + 3] != 0).any())
                L.check(L.lib.brov_set_vehicle_params(self._h, soa.data_ptr(), soa.shape[1], int(cur)))
            yield
        finally:
            self.set_physical(self.phys)
            if self._pv is None:
                L.check(L.lib.brov_set_vehicle_params(self._h, None, 0, 0))
            else:
                L.check(L.lib.brov_set_vehicle_params(self._h, self._pv.data_ptr(), self._pv.shape[1],
                                                      int(self._pv_current)))

    def set_wrench_lag1(self, enable: bool, T_lag: Optional[float] = None) -> None:
        """First-order wrench lag tau_dot = (tau_cmd - tau)/T_lag (extension; wrench models only)."""
        L.check(L.lib.brov_set_wrench_lag1(self._h, int(bool(enable))))
        self._lag1 = bool(enable)
        if T_lag is not None:
            self.phys[L.PH_TLAG1] = float(T_lag)
            self.set_physical(self.phys)

    def set_di_gains(self, K_lin: np.ndarray, K_ang: np.ndarray) -> None:
        """Gains of the double-integrator model as `estimate_di_gains` returns them: v_dot = u K_lin, w_dot = u K_ang,
        both [NU, 3]."""
        K_lin = np.ascontiguousarray(K_lin, dtype=np.float64)
        K_ang = np.ascontiguousarray(K_ang, dtype=np.float64)
        if K_lin.shape != (self.nu, 3) or K_ang.shape != (self.nu, 3):
            raise ValueError(f"K_lin and K_ang must have shape ({self.nu}, 3)")
        L.check(L.lib.brov_set_di_gains(self._h, L.dptr(K_lin), L.dptr(K_ang)))

    def set_allocation(self, alloc: np.ndarray) -> None:
        a = np.ascontiguousarray(alloc, dtype=np.float64).reshape(6, 8)
        L.check(L.lib.brov_set_allocation(self._h, L.dptr(a)))
        self._alloc = a.copy()

    def set_lag_discrete(self, dt: float, Ad: np.ndarray, Bd: np.ndarray) -> None:
        """Override the native ZOH for one dt (e.g. with scipy.signal.cont2discrete's result)."""
        Ad = np.ascontiguousarray(Ad, dtype=np.float64).reshape(3, 3)
        Bd = np.ascontiguousarray(Bd, dtype=np.float64).reshape(3)
        L.check(L.lib.brov_set_lag_discrete(self._h, float(dt), L.dptr(Ad), L.dptr(Bd)))

    # ------------------------------------------------------------------ helpers
    def tensor(self, a, shape=None) -> torch.Tensor:
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        t = t.to(device=self.device, dtype=self.tdtype).contiguous()
        return t if shape is None else t.reshape(shape)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_rows(self, t: torch.Tensor, cols: int, what: str) -> None:
        if t.dim() != 2 or t.shape[1] != cols:
            raise ValueError(f"{what} must have shape [N, {cols}], got {tuple(t.shape)}")

    def _check_lag_inout(self, lag, n: int, per_row: int) -> None:
        """An in/out lag buffer is handed to the library as a raw pointer: it must already be what the kernel expects."""
        if lag is None:
            return
        if (not isinstance(lag, torch.Tensor) or lag.device != self.device or lag.dtype != self.tdtype
                or not lag.is_contiguous() or lag.numel() != n * per_row):
            raise ValueError(f"lag must be a contiguous {self.tdtype} tensor on {self.device} with N*{per_row} elements")

    # ------------------------------------------------------------------ device API
    def rhs(self, x, u, lag: Optional[torch.Tensor] = None, dt: float = 0.02) -> torch.Tensor:
        """xdot for N vehicles (`rov.dynamics(x, u, dt)`).  For the thruster model `lag` [N,24] is advanced in place
        by one ThrusterLag.step, as a reference call does; None = zero lag state, nothing carried."""
        x = self.tensor(x)
        u = self.tensor(u)
        self._check_rows(x, self.nx, "x")
        self._check_rows(u, self.nu, "u")
        n = x.shape[0]
        if u.shape[0] != n:
            raise ValueError("x and u disagree on N")
        self._check_lag_inout(lag, n, self.nlag)
        out = torch.empty((n, self.nx + (6 if self._lag1 else 0)), device=self.device, dtype=self.tdtype)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_rhs(self._h, n, x.data_ptr(), u.data_ptr(), lag.data_ptr() if lag is not None else None,
                                   float(dt), out.data_ptr(), self._stream()))
        return out

    def thruster_wrench(self, u, lag: Optional[torch.Tensor] = None, dt: float = 0.02) -> torch.Tensor:
        """Body wrench of the thruster map (`rov.compute_thruster_forces(u, dt)`), lag advanced in place."""
        u = self.tensor(u)
        self._check_rows(u, 8, "u")
        n = u.shape[0]
        self._check_lag_inout(lag, n, 24)
        out = torch.empty((n, 6), device=self.device, dtype=self.tdtype)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_thruster_wrench(self._h, n, u.data_ptr(), lag.data_ptr() if lag is not None else None,
                                               float(dt), out.data_ptr(), self._stream()))
        return out

    def thruster_wrench_series(self, U, lag0=None, dt: float = 0.02):
        """Body wrench of every row of an input series U [T,8] under ONE lag state carried from row to row — the loop
        `[rov.compute_thruster_forces(u, dt) for u in U]` as one launch.  Returns (tau [T,6], lag_end [24])."""
        U = self.tensor(U)
        self._check_rows(U, 8, "U")
        T_ = U.shape[0]
        l0 = self.tensor(lag0).reshape(24) if lag0 is not None else None
        tau = torch.empty((T_, 6), device=self.device, dtype=self.tdtype)
        lag_end = torch.zeros(24, device=self.device, dtype=self.tdtype) if l0 is None else l0.clone()
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_thruster_wrench_series(self._h, T_, U.data_ptr(), l0.data_ptr() if l0 is not None else None,
                                                      float(dt), tau.data_ptr(), lag_end.data_ptr(), self._stream()))
        return tau, lag_end

    def rhs_host(self, x: np.ndarray, u: np.ndarray, lag: Optional[np.ndarray] = None, dt: float = 0.02) -> np.ndarray:
        """`rhs` with numpy arrays in host memory (engine dtype): one pinned staging copy each way inside the library,
        no torch tensors — the low-latency path behind the model mirrors' per-call `dynamics()`.  `lag` [N,24]
        (thruster model) is advanced in place."""
        x = np.ascontiguousarray(x, dtype=self.ndtype).reshape(-1, self.nx)
        u = np.ascontiguousarray(u, dtype=self.ndtype).reshape(-1, self.nu)
        if u.shape[0] != x.shape[0]:
            raise ValueError("x and u must have the same number of rows")
        if lag is not None and (lag.dtype != self.ndtype or not lag.flags.c_contiguous or lag.size != x.shape[0] * 24):
            raise ValueError(f"lag must be a C-contiguous {np.dtype(self.ndtype)} array with 24 values per row")
        out = np.empty((x.shape[0], self.nx + (6 if self._lag1 else 0)), dtype=self.ndtype)
        L.check(L.lib.brov_rhs_host(self._h, x.shape[0], x.ctypes.data, u.ctypes.data,
                                    lag.ctypes.data if lag is not None else None, float(dt), out.ctypes.data))
        return out

    def thruster_wrench_host(self, u: np.ndarray, lag: Optional[np.ndarray] = None, dt: float = 0.02) -> np.ndarray:
        """`thruster_wrench` with numpy arrays in host memory; `lag` [N,24] is advanced in place."""
        u = np.ascontiguousarray(u, dtype=self.ndtype).reshape(-1, 8)
        if lag is not None and (lag.dtype != self.ndtype or not lag.flags.c_contiguous or lag.size != u.shape[0] * 24):
            raise ValueError(f"lag must be a C-contiguous {np.dtype(self.ndtype)} array with 24 values per row")
        out = np.empty((u.shape[0], 6), dtype=self.ndtype)
        L.check(L.lib.brov_thruster_wrench_host(self._h, u.shape[0], u.ctypes.data,
                                                lag.ctypes.data if lag is not None else None, float(dt), out.ctypes.data))
        return out

    def rollout(self, x0, U=None, dt: float = 0.02, integrator: str = "rk4", lag0=None, stride: int = 0,
                u_layout: str = "auto", step0: int = 0, xT_out: Optional[torch.Tensor] = None,
                lag_out: Optional[torch.Tensor] = None, traj_out: Optional[torch.Tensor] = None,
                want_lag: bool = True, lag_repr: str = "thruster", time_slices: int = 0,
                gen: Optional[InputGenerator] = None, steps: Optional[int] = None, gen_state=None,
                gen_state_out: Optional[torch.Tensor] = None, health: bool = False,
                min_abs_cos: Optional[torch.Tensor] = None, min_abs_cos_accumulate: bool = False,
                singular_eps: float = 0.0) -> RolloutResult:
        """Open-loop rollout of N vehicles (`simulate_physics` batched).

        x0 [N,NX]; U is one of
          [T,N,NU]  per-vehicle series, time-major     (u_layout "tnc")
          [T,NU]    one series shared by every vehicle (u_layout "shared")
          [N,NU]    one constant input per vehicle     (u_layout "const", needs `steps` via U.shape... see below)
        With u_layout="auto" a 3-D U is "tnc" and a 2-D U is "shared".  For "const" pass U=(tensor [N,NU], steps).
        stride > 0 stores the state after every stride-th step into traj [T//stride, N, NX].

        gen=InputGenerator(...), steps=T: the inputs are generated inside the kernel (U is not used); gen_state
        [N,NU] is the AR(1) state to continue from (None = zeros), the state after the call comes back as
        result.gen_state (written into gen_state_out if given; may be the same tensor).

        Thruster model: lag_repr="thruster" (default) exchanges the per-thruster lag states [N,24] — the reference's
        hidden state `ThrusterLag._x`; lag_repr="projected" exchanges the allocation-projected states [N,18] (see
        include/brov.h) — what the kernels integrate, the cheapest carry between the chunks of a long rollout.

        health=True returns int64 [2] counts (non-finite final states, vehicles that came within singular_eps of
        theta = +-pi/2); min_abs_cos [N] (in/out with min_abs_cos_accumulate) is the per-vehicle running minimum of
        |cos theta|.
        """
        x0 = self.tensor(x0)
        self._check_rows(x0, self.nx, "x0")
        n = x0.shape[0]
        Ut = None
        if gen is not None:
            if steps is None:
                raise ValueError("generated inputs need steps=")
            steps, st, sn = int(steps), 0, 0
        elif u_layout == "const":
            Ut, steps = U
            Ut = self.tensor(Ut)
            self._check_rows(Ut, self.nu, "U")
            st, sn = 0, self.nu
        else:
            Ut = self.tensor(U)
            if u_layout == "auto":
                u_layout = "tnc" if Ut.dim() == 3 else "shared"
            if u_layout == "tnc":
                if Ut.dim() != 3 or Ut.shape[1] != n or Ut.shape[2] != self.nu:
                    raise ValueError(f"U must have shape [T, {n}, {self.nu}], got {tuple(Ut.shape)}")
                st, sn = n * self.nu, self.nu
            elif u_layout == "shared":
                self._check_rows(Ut, self.nu, "U")
                st, sn = self.nu, 0
            else:
                raise ValueError("u_layout must be auto|tnc|shared|const")
            steps = Ut.shape[0]
        integ = INTEGRATORS[integrator]
        xT = xT_out if xT_out is not None else torch.empty_like(x0)
        if lag_repr not in ("thruster", "projected"):
            raise ValueError("lag_repr must be 'thruster' or 'projected'")
        proj = lag_repr == "projected" and self.model == "thruster8"
        nlag = 18 if proj else self.nlag
        lag_in = None
        if nlag and lag0 is not None:
            lag_in = self.tensor(lag0).reshape(n, nlag)
        if nlag and want_lag and lag_out is None:
            lag_out = torch.empty((n, nlag), device=self.device, dtype=self.tdtype)
        if nlag and lag_out is not None:
            self._check_lag_inout(lag_out, n, nlag)
        traj = traj_out
        if stride and traj is None:
            nsnap = (step0 + steps) // stride - step0 // stride
            traj = torch.empty((nsnap, n, self.nx), device=self.device, dtype=self.tdtype)
        d = L.RolloutDesc()
        d.struct_size = C.sizeof(L.RolloutDesc)
        d.integrator = integ
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.x0_dev, d.xT_dev = x0.data_ptr(), xT.data_ptr()
        d.u_dev = Ut.data_ptr() if Ut is not None else None
        d.u_stride_t, d.u_stride_n = st, sn
        d.lag_in_dev = lag_in.data_ptr() if lag_in is not None else None
        d.lag_out_dev = lag_out.data_ptr() if (nlag and lag_out is not None) else None
        d.traj_dev = traj.data_ptr() if (stride and traj is not None and traj.numel()) else None
        d.stride = max(int(stride), 1)
        d.step0 = int(step0)
        d.snap_base = int(step0) // max(int(stride), 1)
        d.lag_in_repr = d.lag_out_repr = L.LAG_PROJECTED if proj else L.LAG_THRUSTER
        d.time_slices = int(time_slices)  # 0 = automatic temporal tiling (bit-identical results for every value)
        gs_in = gs_out = None
        if gen is not None:
            if gen_state is not None:
                gs_in = self.tensor(gen_state).reshape(n, self.nu)
            gs_out = gen_state_out if gen_state_out is not None else torch.empty((n, self.nu), device=self.device, dtype=self.tdtype)
            self._check_lag_inout(gs_out, n, self.nu)
            gen.fill(d.gen, self.nu, gs_in.data_ptr() if gs_in is not None else None, gs_out.data_ptr())
        hc = None
        if health:
            hc = torch.zeros(2, device=self.device, dtype=torch.int64)
            d.health_dev = hc.data_ptr()
        if min_abs_cos is not None:
            self._check_lag_inout(min_abs_cos, n, 1)
            d.min_abs_cos_dev = min_abs_cos.data_ptr()
            d.min_abs_cos_accumulate = int(bool(min_abs_cos_accumulate))
        d.singular_eps = float(singular_eps)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_rollout(self._h, C.byref(d), self._stream()))
        return RolloutResult(xT=xT, lag=lag_out if (nlag and want_lag) else None, traj=traj if stride else None,
                             gen_state=gs_out, health=hc, min_abs_cos=min_abs_cos)

    def generate_inputs(self, gen: InputGenerator, steps: int, step0: int = 0, first: int = 0, vstride: int = 1,
                        n_sel: int = 1, state_in=None):
        """The command signal the kernels generate, as an array: (U [steps, n_sel, NU], state_out [n_sel, NU]) for the
        vehicles first, first + vstride, ... and steps step0 .. step0 + steps - 1 (brov_generate_inputs).  Feeding U to
        `rollout` reproduces the generated-input rollout of those vehicles bit for bit; a CPU reference consumes the
        same numbers."""
        out = torch.empty((int(steps), int(n_sel), self.nu), device=self.device, dtype=self.tdtype)
        so = torch.empty((int(n_sel), self.nu), device=self.device, dtype=self.tdtype)
        si = self.tensor(state_in).reshape(n_sel, self.nu) if state_in is not None else None
        d = L.GenInputsDesc()
        d.struct_size = C.sizeof(L.GenInputsDesc)
        d.dtype, d.nu, d.device = self._code, self.nu, self.device_index
        d.first, d.vstride, d.n_sel = int(first), int(vstride), int(n_sel)
        d.step0, d.steps = int(step0), int(steps)
        gen.fill(d.gen, self.nu, si.data_ptr() if si is not None else None, so.data_ptr())
        d.out_dev = out.data_ptr()
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_generate_inputs(C.byref(d), self._stream()))
        return out, so

    def project_lag(self, lag24) -> torch.Tensor:
        """Per-thruster lag states [N,8,3] -> allocation-projected states [N,18] (Z[c][k] = sum_i alloc[c][i] lag[i][k])."""
        if self._alloc is None:
            raise ValueError("project_lag applies to the thruster model")
        A = self.tensor(self._alloc)     # the allocation the kernels use (set_allocation keeps it current)
        return torch.einsum("ci,nik->nck", A, self.tensor(lag24).reshape(-1, 8, 3)).reshape(-1, 18).contiguous()

    def step(self, x, u, lag=None, dt: float = 0.02, integrator: str = "rk4") -> RolloutResult:
        """One integrator step for N vehicles (u [N,NU]) through brov_step; `lag` [N,NLAG] is advanced in place."""
        x = self.tensor(x)
        u = self.tensor(u)
        self._check_rows(x, self.nx, "x")
        self._check_rows(u, self.nu, "u")
        n = x.shape[0]
        if u.shape[0] != n:
            raise ValueError("x and u must have the same number of rows")
        lag_t = None
        if self.nlag and lag is not None:
            lag_t = self.tensor(lag).reshape(n, self.nlag)
            self._check_lag_inout(lag_t, n, self.nlag)
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_step(self._h, INTEGRATORS[integrator], n, x.data_ptr(), u.data_ptr(), float(dt),
                                    out.data_ptr(), lag_t.data_ptr() if lag_t is not None else None, self._stream()))
        return RolloutResult(xT=out, lag=lag_t, traj=None)

    def carry_steps(self, dt: float = 0.02, integrator: str = "rk4") -> int:
        """Replay depth (integrator steps) of the carried-lag evaluator for this dt / integrator."""
        out = C.c_longlong()
        L.check(L.lib.brov_se_carry_steps(self._h, float(dt), INTEGRATORS[integrator], C.byref(out)))
        return int(out.value)

    def multistep_se(self, X, U, horizons: Sequence[int], dt: float = 0.02, integrator: str = "rk4",
                     lag0=None, n_windows: Optional[int] = None, lag_mode: str = "reset", window0: int = 0,
                     row0: int = 0, se_out: Optional[torch.Tensor] = None, health_out: Optional[torch.Tensor] = None,
                     singular_eps: float = 0.0, workspace: Optional[torch.Tensor] = None, time_slices: int = 0):
        """Sum of squared endpoint errors per horizon over sliding windows of one recorded series.
        Returns (se [MAX_H] float64 device tensor, counts list).  See brov_multistep_se in include/brov.h.
        lag_mode="carry" (thruster model, one horizon): the reference's literal semantics — the lag state left by
        windows 0..k-1 is what window k starts from.  window0 / row0: global indices of the first local window / row
        when X, U are a shard of a longer series.
        se_out: float64 [MAX_H] device tensor to write into (e.g. a slice of a reduction buffer); health_out: int64 [2]
        device tensor receiving the number of windows with a non-finite endpoint error / that came within
        singular_eps of theta = +-pi/2.
        workspace: uint8 device tensor of at least brov_se_workspace_bytes(n_windows) for the per-block partial sums
        (default: the engine's own, which calls on DIFFERENT streams must not share)."""
        X = self.tensor(X)
        U = self.tensor(U)
        self._check_rows(X, self.nx, "X")
        self._check_rows(U, self.nu, "U")
        rows = X.shape[0]
        if U.shape[0] != rows:
            raise ValueError("X and U must have the same number of rows")
        hs = [int(h) for h in horizons]
        if not 1 <= len(hs) <= L.MAX_H or any(h < 1 for h in hs) or sorted(set(hs)) != hs:
            raise ValueError(f"horizons must be 1..{L.MAX_H} strictly ascending positive integers")
        if lag_mode not in ("reset", "carry"):
            raise ValueError("lag_mode must be 'reset' or 'carry'")
        carry = lag_mode == "carry" and self.model == "thruster8"
        off = int(window0) - int(row0)
        nwin = max(rows - off - hs[0], 0) if n_windows is None else int(n_windows)
        nbytes = L.lib.brov_se_workspace_bytes(nwin)
        if workspace is not None:
            if workspace.dtype != torch.uint8 or workspace.device != self.device or workspace.numel() < nbytes:
                raise ValueError(f"workspace must be a uint8 tensor of at least {nbytes} bytes on {self.device}")
            ws = workspace
        else:
            if self._ws is None or self._ws.numel() < nbytes:
                self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            ws = self._ws
        if se_out is None:
            se = torch.zeros(L.MAX_H, dtype=torch.float64, device=self.device)
        else:
            se = se_out
            if se.dtype != torch.float64 or se.device != self.device or not se.is_contiguous() or se.numel() < L.MAX_H:
                raise ValueError(f"se_out must be a contiguous float64 tensor with {L.MAX_H} elements on {self.device}")
        counts = (C.c_longlong * L.MAX_H)()
        d = L.SeDesc()
        d.struct_size = C.sizeof(L.SeDesc)
        d.integrator = INTEGRATORS[integrator]
        d.rows, d.n_windows, d.dt = rows, nwin, float(dt)
        d.X_dev, d.U_dev = X.data_ptr(), U.data_ptr()
        lag_t = None
        if lag0 is not None:
            lag_t = self.tensor(lag0).reshape(nwin, 24)
        d.lag0_dev = lag_t.data_ptr() if lag_t is not None else None
        d.n_horizons = len(hs)
        for i, h in enumerate(hs):
            d.horizons[i] = h
        d.se_out_dev = se.data_ptr()
        d.count_out = counts
        d.workspace_dev = ws.data_ptr()
        d.workspace_bytes = nbytes
        d.lag_carry = int(carry)
        d.time_slices = int(time_slices)      # 0: automatic (against the partial last wave), 1: off, 2..4: forced
        d.window0, d.row0 = (int(window0), int(row0)) if carry else (0, 0)
        if health_out is not None:
            if health_out.dtype != torch.int64 or health_out.device != self.device or health_out.numel() < 2:
                raise ValueError("health_out must be an int64 tensor with 2 elements on the engine's device")
            d.health_dev = health_out.data_ptr()
            d.singular_eps = float(singular_eps)
        if not carry and off:
            raise ValueError("window0 != row0 needs lag_mode='carry'")
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_multistep_se(self._h, C.byref(d), self._stream()))
        return se, [int(counts[i]) for i in range(len(hs))]

    def multistep_rmse(self, X, U, horizons, dt: float = 0.02, integrator: str = "rk4", lag0=None,
                       lag_mode: str = "reset"):
        """RMSE per horizon, `sqrt(se / (n_windows * n_states))`, NaN where no window fits (reference semantics).
        lag_mode="reset": every window starts from `lag0` (default zero), all horizons share one pass.
        lag_mode="carry": thruster-lag state carried from window to window as in the reference (one pass per horizon)."""
        single = np.isscalar(horizons)
        hs = [int(horizons)] if single else [int(h) for h in horizons]
        order = sorted(set(hs))
        out = {}
        group = 1 if (lag_mode == "carry" and self.model == "thruster8") else L.MAX_H
        X = self.tensor(X)
        U = self.tensor(U)
        for i in range(0, len(order), group):
            part = order[i:i + group]
            se, cnt = self.multistep_se(X, U, part, dt, integrator, lag0, lag_mode=lag_mode)
            se = se.cpu().numpy()
            for j, h in enumerate(part):
                out[h] = float(np.sqrt(se[j] / (cnt[j] * self.nx))) if cnt[j] > 0 else float("nan")
        return out[hs[0]] if single else [out[h] for h in hs]

    def multistep_se_sweep(self, X, U, horizons: Sequence[int], phys_table: np.ndarray, dt: float = 0.02,
                           integrator: str = "rk4", lag_mode: str = "reset", lag0=None,
                           health_out: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None,
                           singular_eps: float = 0.0, workspace_cap: int = SWEEP_WORKSPACE_CAP):
        """`multistep_se` for P candidate vehicles against one recorded series (brov_multistep_se_sweep).
        phys_table [P, NPHYS]: one physical vector per candidate (derived row by row as set_vehicle_physical does; see
        with_minv for tables that perturb the masses).  The engine's own coefficients are not used; allocation and lag
        discretisation are the engine's.  Returns (se [P, MAX_H] float64 device tensor, counts list): row c equals
        `set_physical(phys_table[c])` + `multistep_se(..., time_slices=1)`.
        lag_mode="carry" (thruster model, one horizon): the carried lag each window starts from is computed once for all
        candidates.  lag0 [n_windows, 24] (reset mode) is shared by every candidate.  health_out: int64 [P, 2] device
        tensor receiving, per candidate, the windows with a non-finite endpoint error / that came within singular_eps of
        theta = +-pi/2.  The candidates are split over several launches so that the workspace stays within
        workspace_cap bytes (a workspace passed in must hold one launch: brov_se_sweep_workspace_bytes)."""
        X = self.tensor(X)
        U = self.tensor(U)
        self._check_rows(X, self.nx, "X")
        self._check_rows(U, self.nu, "U")
        rows = X.shape[0]
        if U.shape[0] != rows:
            raise ValueError("X and U must have the same number of rows")
        hs = [int(h) for h in horizons]
        if not 1 <= len(hs) <= L.MAX_H or any(h < 1 for h in hs) or sorted(set(hs)) != hs:
            raise ValueError(f"horizons must be 1..{L.MAX_H} strictly ascending positive integers")
        if lag_mode not in ("reset", "carry"):
            raise ValueError("lag_mode must be 'reset' or 'carry'")
        carry = lag_mode == "carry" and self.model == "thruster8"
        ph = np.asarray(phys_table, dtype=np.float64)
        if ph.ndim != 2 or ph.shape[1] != L.NPHYS:
            raise ValueError(f"phys_table must have shape [P, {L.NPHYS}]")
        P = ph.shape[0]
        kp = derive_params(ph)                                                   # [P, NKP]
        # one flag for the whole table: a split sweep runs the same kernel build in every launch
        any_current = int(bool(np.any(ph[:, L.PH_CURRENT:L.PH_CURRENT + 3] != 0.0)))
        nwin = max(rows - hs[0], 0)
        per_launch = P
        while per_launch > 1 and L.lib.brov_se_sweep_workspace_bytes(per_launch, nwin, int(carry)) > workspace_cap:
            per_launch = (per_launch + 1) // 2
        nbytes = L.lib.brov_se_sweep_workspace_bytes(max(per_launch, 1), nwin, int(carry))
        if workspace is not None:
            if workspace.dtype != torch.uint8 or workspace.device != self.device or workspace.numel() < nbytes:
                raise ValueError(f"workspace must be a uint8 tensor of at least {nbytes} bytes on {self.device}")
            ws = workspace
        else:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        if health_out is not None and (health_out.dtype != torch.int64 or health_out.device != self.device
                                       or not health_out.is_contiguous() or health_out.numel() != 2 * P):
            raise ValueError(f"health_out must be a contiguous int64 tensor with {2 * P} elements on {self.device}")
        lag_t = self.tensor(lag0).reshape(nwin, 24) if (lag0 is not None and self.model == "thruster8") else None
        se = torch.zeros((P, L.MAX_H), dtype=torch.float64, device=self.device)
        counts = (C.c_longlong * L.MAX_H)()
        d = L.SeSweepDesc()
        d.struct_size = C.sizeof(L.SeSweepDesc)
        d.integrator = INTEGRATORS[integrator]
        d.rows, d.n_windows, d.dt = rows, nwin, float(dt)
        d.X_dev, d.U_dev = X.data_ptr(), U.data_ptr()
        d.lag0_dev = lag_t.data_ptr() if lag_t is not None else None
        d.n_horizons = len(hs)
        for i, h in enumerate(hs):
            d.horizons[i] = h
        d.lag_carry = int(carry)
        d.any_current = any_current
        d.count_out = counts
        d.singular_eps = float(singular_eps)
        d.workspace_dev, d.workspace_bytes = ws.data_ptr(), ws.numel()
        with torch.cuda.device(self.device):
            for lo in range(0, max(P, 1), max(per_launch, 1)):
                hi = min(P, lo + per_launch)
                soa = torch.from_numpy(np.ascontiguousarray(kp[lo:hi].T)).to(self.device, self.tdtype).contiguous()
                d.n_candidates = hi - lo
                d.kp_soa_dev = soa.data_ptr() if hi > lo else None
                d.se_out_dev = se[lo:hi].data_ptr() if hi > lo else None
                d.health_dev = health_out.reshape(P, 2)[lo:hi].data_ptr() if (health_out is not None and hi > lo) else None
                L.check(L.lib.brov_multistep_se_sweep(self._h, C.byref(d), self._stream()))
        return se, [int(counts[i]) for i in range(len(hs))]

    def multistep_rmse_sweep(self, X, U, horizons, phys_table: np.ndarray, dt: float = 0.02, integrator: str = "rk4",
                             lag_mode: str = "reset", lag0=None) -> np.ndarray:
        """RMSE per candidate and horizon, numpy [P, len(horizons)] (`multistep_rmse` for every row of phys_table;
        NaN where no window fits).  lag_mode="carry" (thruster model) runs one pass per horizon."""
        single = np.isscalar(horizons)
        hs = [int(horizons)] if single else [int(h) for h in horizons]
        order = sorted(set(hs))
        P = np.shape(phys_table)[0]
        out = {}
        group = 1 if (lag_mode == "carry" and self.model == "thruster8") else L.MAX_H
        X = self.tensor(X)
        U = self.tensor(U)
        for i in range(0, len(order), group):
            part = order[i:i + group]
            se, cnt = self.multistep_se_sweep(X, U, part, phys_table, dt, integrator, lag_mode=lag_mode, lag0=lag0)
            se = se.cpu().numpy()
            for j, h in enumerate(part):
                out[h] = np.sqrt(se[:, j] / (cnt[j] * self.nx)) if cnt[j] > 0 else np.full(P, np.nan)
        return np.stack([out[h] for h in hs], axis=1) if P else np.zeros((0, len(hs)))

    def multistep_se_grad(self, X, U, horizons: Sequence[int], phys: np.ndarray, params, dt: float = 0.02,
                          integrator: str = "rk4", lag_mode: str = "reset", lag0=None, rebuild_minv: bool = True,
                          health_out: Optional[torch.Tensor] = None, singular_eps: float = 0.0,
                          n_windows: Optional[int] = None, window0: int = 0, row0: int = 0) -> GradResult:
        """`multistep_se` of the vehicle `phys` together with its exact gradient and Gauss-Newton matrix in the
        selected physical parameters (brov_multistep_se_grad; forward-mode sensitivities through every integrator
        step).  params: PH_* indices, attribute names or groups (see parameter_indices); the coefficient directions
        come from coefficient_directions(phys, params, rebuild_minv), the point is derive_params(with_minv(phys)) (or
        of phys itself without rebuild_minv).  The engine's own coefficients are not used.  fp64 engines only.
        lag_mode="carry" (thruster model) makes one call per horizon, as multistep_rmse does.  health_out: int64 [2]
        device tensor (accumulated over the calls of a carried-lag evaluation).  window0 / row0 / n_windows: a shard
        of a longer series, as in multistep_se."""
        X = self.tensor(X)
        U = self.tensor(U)
        self._check_rows(X, self.nx, "X")
        self._check_rows(U, self.nu, "U")
        rows = X.shape[0]
        if U.shape[0] != rows:
            raise ValueError("X and U must have the same number of rows")
        hs = [int(h) for h in horizons]
        if not 1 <= len(hs) <= L.MAX_H or any(h < 1 for h in hs) or sorted(set(hs)) != hs:
            raise ValueError(f"horizons must be 1..{L.MAX_H} strictly ascending positive integers")
        if lag_mode not in ("reset", "carry"):
            raise ValueError("lag_mode must be 'reset' or 'carry'")
        carry = lag_mode == "carry" and self.model == "thruster8"
        off = int(window0) - int(row0)
        if off and not carry:
            raise ValueError("window0 != row0 needs lag_mode='carry'")
        ph = np.asarray(phys, dtype=np.float64).reshape(L.NPHYS)
        idx = parameter_indices(params)
        dirs = coefficient_directions(ph, idx, rebuild_minv)
        kp = derive_params(with_minv(ph) if rebuild_minv else ph)
        p = len(idx)
        any_current = int(bool(np.any(kp[KP_CUR:KP_CUR + 3] != 0.0) or np.any(dirs[:, KP_CUR:KP_CUR + 3] != 0.0)))
        kp_t = torch.as_tensor(kp, dtype=torch.float64, device=self.device)
        dirs_t = torch.as_tensor(np.ascontiguousarray(dirs), dtype=torch.float64, device=self.device)
        if health_out is not None:
            if health_out.dtype != torch.int64 or health_out.device != self.device or health_out.numel() != 2:
                raise ValueError("health_out must be an int64 tensor with 2 elements on the engine's device")
        groups = [[h] for h in hs] if carry else [hs]
        se = torch.zeros((len(hs),), dtype=torch.float64, device=self.device)
        grad = torch.zeros((len(hs), p), dtype=torch.float64, device=self.device)
        gn = torch.zeros((len(hs), p, p), dtype=torch.float64, device=self.device)
        counts = []
        hc = health_out
        if health_out is not None and carry:      # one count over the per-horizon calls
            health_out.zero_()
            hc = torch.zeros(2, dtype=torch.int64, device=self.device)
        for g in groups:
            nwin = max(rows - off - g[0], 0) if n_windows is None else int(n_windows)
            nbytes = L.lib.brov_se_grad_workspace_bytes(nwin, p, int(carry))
            ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
            se_o = torch.zeros(L.MAX_H, dtype=torch.float64, device=self.device)
            gr_o = torch.zeros((L.MAX_H, p), dtype=torch.float64, device=self.device)
            gn_o = torch.zeros((L.MAX_H, p, p), dtype=torch.float64, device=self.device)
            cnt = (C.c_longlong * L.MAX_H)()
            d = L.SeGradDesc()
            d.struct_size = C.sizeof(L.SeGradDesc)
            d.integrator = INTEGRATORS[integrator]
            d.rows, d.n_windows, d.dt = rows, nwin, float(dt)
            d.X_dev, d.U_dev = X.data_ptr(), U.data_ptr()
            lag_t = self.tensor(lag0).reshape(nwin, 24) if (lag0 is not None and self.model == "thruster8") else None
            d.lag0_dev = lag_t.data_ptr() if lag_t is not None else None
            d.n_horizons = len(g)
            for i, h in enumerate(g):
                d.horizons[i] = h
            d.lag_carry = int(carry)
            d.window0, d.row0 = (int(window0), int(row0)) if carry else (0, 0)
            d.kp_dev, d.any_current, d.n_dirs, d.dirs_dev = kp_t.data_ptr(), any_current, p, dirs_t.data_ptr()
            d.se_out_dev, d.grad_out_dev, d.gn_out_dev = se_o.data_ptr(), gr_o.data_ptr(), gn_o.data_ptr()
            d.count_out = cnt
            d.health_dev = hc.data_ptr() if hc is not None else None
            d.singular_eps = float(singular_eps)
            d.workspace_dev, d.workspace_bytes = ws.data_ptr(), nbytes
            with torch.cuda.device(self.device):
                L.check(L.lib.brov_multistep_se_grad(self._h, C.byref(d), self._stream()))
            if carry and health_out is not None:
                health_out += hc
            at = hs.index(g[0])
            se[at:at + len(g)] = se_o[:len(g)]
            grad[at:at + len(g)] = gr_o[:len(g)]
            gn[at:at + len(g)] = gn_o[:len(g)]
            counts += [int(cnt[i]) for i in range(len(g))]
        return GradResult(se=se, grad=grad, gn=gn, counts=counts, names=[PHYS_NAMES[i] for i in idx], index=idx)

    @property
    def nz(self) -> int:
        """Length of the augmented state z that linearize differentiates: x, plus the projected lag [18] (thruster)."""
        return self.nx + (18 if self.model == "thruster8" else 0)

    def linearize(self, x0, U, dt: float = 0.02, integrator: str = "rk4", lag0=None, lag_repr: str = "thruster",
                  u_layout: str = "auto", want_traj: bool = True, health: bool = False,
                  jac_out: Optional[torch.Tensor] = None, singular_eps: float = 0.0) -> LinearizeResult:
        """Exact Jacobians of the discrete step along N trajectories (brov_linearize): for every step k and vehicle i,
        A[k, i] = dPhi/dz and B[k, i] = dPhi/du at (z_k, u_k), where z_{k+1} = Phi(z_k, u_k) is one integrator step.

        z = [x | Z]: for the thruster model Z [18] is the allocation-projected lag Z[c][k] = sum_i alloc[c][i] L[i][k]
        (project_lag), the only form in which the dynamics see the lag; the result is ALWAYS in these projected
        coordinates (NZ = 30), and per-thruster Jacobians follow by the chain rule with Z = P L.  Wrench models: z = x.
        lag0 (thruster model): per-thruster [N,24] with lag_repr="thruster" (projected here), or projected [N,18] with
        lag_repr="projected"; None = zeros.

        U is one of
          [T,N,NU]  per-vehicle series, time-major   (u_layout "tnc"; the default for a 3-D U)
          [N,NU]    one step with one input per vehicle (the default for a 2-D U; T = 1)
          [T,NU]    one series shared by every vehicle (u_layout "shared")
          (U [N,NU], T) one constant input per vehicle for T steps (u_layout "const")
        The outputs keep the step axis also for T = 1.  A and B are views of one J [T, N, NZ, NZ+NU] (jac_out, if
        given: a contiguous float64 tensor of that shape on the engine's device).  The derivative is that of the
        computed function, branch taken (d|x| = sign(x) dx; the clamped cos(theta) and the quaternion fallback are
        constants).  health=True returns int64 [2] counts of vehicles with a non-finite z or Jacobian entry and of
        vehicles that came within singular_eps (0 = 1e-3) of theta = +-pi/2.  fp64 engines with shared coefficients."""
        x0 = self.tensor(x0)
        self._check_rows(x0, self.nx, "x0")
        n = x0.shape[0]
        if u_layout == "const":
            Ut, steps = U
            Ut = self.tensor(Ut)
            self._check_rows(Ut, self.nu, "U")
            if Ut.shape[0] != n:
                raise ValueError(f"U must have shape [{n}, {self.nu}], got {tuple(Ut.shape)}")
            steps, st, sn = int(steps), 0, self.nu
        else:
            Ut = self.tensor(U)
            if u_layout == "auto":
                u_layout = "tnc" if Ut.dim() == 3 else "step"
            if u_layout == "tnc":
                if Ut.dim() != 3 or Ut.shape[1] != n or Ut.shape[2] != self.nu:
                    raise ValueError(f"U must have shape [T, {n}, {self.nu}], got {tuple(Ut.shape)}")
                steps, st, sn = Ut.shape[0], n * self.nu, self.nu
            elif u_layout == "step":
                if Ut.dim() != 2 or Ut.shape[0] != n or Ut.shape[1] != self.nu:
                    raise ValueError(f"U must have shape [{n}, {self.nu}], got {tuple(Ut.shape)}")
                steps, st, sn = 1, 0, self.nu
            elif u_layout == "shared":
                self._check_rows(Ut, self.nu, "U")
                steps, st, sn = Ut.shape[0], self.nu, 0
            else:
                raise ValueError("u_layout must be auto|tnc|shared|const")
        z0 = self._z0(x0, lag0, lag_repr, n)
        nz, nc = self.nz, self.nz + self.nu
        shape = (steps, n, nz, nc)
        if jac_out is not None:
            if (not isinstance(jac_out, torch.Tensor) or jac_out.device != self.device or jac_out.dtype != torch.float64
                    or not jac_out.is_contiguous() or tuple(jac_out.shape) != shape):
                raise ValueError(f"jac_out must be a contiguous float64 tensor of shape {shape} on {self.device}")
            J = jac_out
        else:
            J = torch.empty(shape, device=self.device, dtype=self.tdtype)
        z = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        zt = torch.empty((steps, n, nz), device=self.device, dtype=self.tdtype) if want_traj else None
        hc = torch.zeros(2, device=self.device, dtype=torch.int64) if health else None
        d = L.LinearizeDesc()
        d.struct_size = C.sizeof(L.LinearizeDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.z0_dev, d.u_dev = z0.data_ptr(), Ut.data_ptr()
        d.u_stride_t, d.u_stride_n = st, sn
        d.z_out_dev = z.data_ptr()
        d.z_traj_dev = zt.data_ptr() if zt is not None else None
        d.jac_dev = J.data_ptr()
        d.health_dev = hc.data_ptr() if hc is not None else None
        d.singular_eps = float(singular_eps)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_linearize(self._h, C.byref(d), self._stream()))
        return LinearizeResult(A=J[..., :nz], B=J[..., nz:], z=z, z_traj=zt, health=hc)

    def _z0(self, x0, lag0, lag_repr: str, n: int):
        """z_0 = [x0 | Z0] of the linearize / adjoint / closed-loop / EKF calls: the thruster model's lag0 per thruster
        [N,24] (lag_repr="thruster", projected here) or projected [N,18] ("projected"), None = zeros; x0 otherwise"""
        if lag_repr not in ("thruster", "projected"):
            raise ValueError("lag_repr must be 'thruster' or 'projected'")
        if self.model != "thruster8":
            return x0
        if lag0 is None:
            Z0 = torch.zeros((n, 18), device=self.device, dtype=self.tdtype)
        elif lag_repr == "thruster":
            Z0 = self.project_lag(self.tensor(lag0).reshape(n, 24))
        else:
            Z0 = self.tensor(lag0).reshape(n, 18)
        return torch.cat([x0, Z0], dim=1).contiguous()

    def _glag0(self, gz0, lag_repr: str, n: int):
        """the lag part of dL/dz_0 in the representation lag0 came in: per thruster P^T gZ0 (Z = P L), or gZ0 itself;
        None for the wrench models"""
        if self.model != "thruster8":
            return None
        gZ0 = gz0[:, self.nx:]
        if lag_repr == "thruster":
            A = self.tensor(self._alloc)
            return torch.einsum("ci,nck->nik", A, gZ0.reshape(n, 6, 3)).reshape(n, 24).contiguous()
        return gZ0

    def _cotangents(self, gtraj, gzT, steps: int, stride: int, n: int, width: int):
        """the trajectory cotangent gtraj [T//stride, N, width] and the terminal one gzT [N, NZ] as tensors (or None),
        their shapes checked"""
        gt = None
        if gtraj is not None:
            gt = self.tensor(gtraj)
            ns = steps // int(stride) if int(stride) >= 1 else None
            if ns is not None and tuple(gt.shape) != (ns, n, width):
                raise ValueError(f"gtraj must have shape [{ns}, {n}, {width}], got {tuple(gt.shape)}")
        gT = None
        if gzT is not None:
            gT = self.tensor(gzT)
            if tuple(gT.shape) != (n, self.nz):
                raise ValueError(f"gzT must have shape [{n}, {self.nz}], got {tuple(gT.shape)}")
        return gt, gT

    def _cost_weights(self, d, cost_q, cost_r):
        """the closed-loop cost weights cost_q [NZ] / cost_r [NU] (scalars broadcast; None leaves them zero) into d.q / d.r"""
        if cost_q is not None:
            q = np.broadcast_to(np.asarray(cost_q, float), (self.nz,))
            for j in range(self.nz):
                d.q[j] = float(q[j])
        if cost_r is not None:
            rw = np.broadcast_to(np.asarray(cost_r, float), (self.nu,))
            for r in range(self.nu):
                d.r[r] = float(rw[r])

    def _inputs(self, U, n: int, u_layout: str):
        """(tensor, steps, stride_t, stride_n) of a rollout input U in the layouts of `rollout`"""
        if u_layout == "const":
            Ut, steps = U
            Ut = self.tensor(Ut)
            if Ut.dim() != 2 or Ut.shape[0] != n or Ut.shape[1] != self.nu:
                raise ValueError(f"U must have shape [{n}, {self.nu}], got {tuple(Ut.shape)}")
            return Ut, int(steps), 0, self.nu
        Ut = self.tensor(U)
        if u_layout == "auto":
            u_layout = "tnc" if Ut.dim() == 3 else "shared"
        if u_layout == "tnc":
            if Ut.dim() != 3 or Ut.shape[1] != n or Ut.shape[2] != self.nu:
                raise ValueError(f"U must have shape [T, {n}, {self.nu}], got {tuple(Ut.shape)}")
            return Ut, Ut.shape[0], n * self.nu, self.nu
        if u_layout == "shared":
            if Ut.dim() != 2 or Ut.shape[1] != self.nu:
                raise ValueError(f"U must have shape [T, {self.nu}], got {tuple(Ut.shape)}")
            return Ut, Ut.shape[0], self.nu, 0
        raise ValueError("u_layout must be auto|tnc|shared|const")

    def rollout_vjp(self, x0, U, gtraj=None, gzT=None, stride: int = 0, dt: float = 0.02, integrator: str = "rk4",
                    lag0=None, lag_repr: str = "thruster", u_layout: str = "auto", health: bool = False,
                    singular_eps: float = 0.0, coef: bool = False) -> VjpResult:
        """Reverse-mode gradients of N rollouts (brov_rollout_vjp): for every vehicle, with
            L = sum_{k = stride, 2 stride, ... <= T} <c_k, x_k> + <g_T, z_T>,
        returns dL/dz_0 (as gx0 and glag0) and dL/du_k for every step, in one launch and without forming the step
        Jacobians.  The step is differentiated as `linearize` differentiates it, so the result equals the chain
        lambda_k = A_k^T lambda_{k+1} + c_k, gu_k = B_k^T lambda_{k+1} over linearize's Jacobians to rounding.

        gtraj [T//stride, N, NX]: the cotangents c_k, in the layout of rollout's traj (None: no trajectory term);
        gzT [N, NZ]: the terminal cotangent on z_T = [x_T | Z_T] (projected lag for the thruster model; None: zero).
        U as in `rollout` ([T,N,NU] "tnc", [T,NU] "shared", (U [N,NU], T) "const"); gU is always [T, N, NU].
        lag0 (thruster model): per-thruster [N,24] with lag_repr="thruster", projected [N,18] with "projected";
        glag0 comes back in the same representation (per thruster: P^T gZ0 by the chain rule with Z = P L).
        The call allocates its workspace, T * N * NZ doubles; split longer horizons as include/brov.h describes.
        fp64 engines with shared coefficients.
        coef=True (brov_rollout_vjp_coef): also returns gkp [N, NKP], dL/dkp of each vehicle's kernel coefficients
        (derive_params layout; the lag entries are 0), and accepts a per-vehicle table (set_vehicle_physical) of N
        rows; with shared coefficients their gradient is gkp.sum(0).  gx0, glag0 and gU are those of coef=False."""
        x0 = self.tensor(x0)
        self._check_rows(x0, self.nx, "x0")
        n = x0.shape[0]
        Ut, steps, st, sn = self._inputs(U, n, u_layout)
        z0 = self._z0(x0, lag0, lag_repr, n)
        nz = self.nz
        gt, gT = self._cotangents(gtraj, gzT, steps, stride, n, self.nx)
        gz0 = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        gU = torch.empty((steps, n, self.nu), device=self.device, dtype=self.tdtype)
        z = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        wsb = int(L.lib.brov_rollout_vjp_workspace_bytes(MODELS[self.model], n, steps))
        ws = torch.empty((max(wsb, 8) + 7) // 8, device=self.device, dtype=torch.float64)
        hc = torch.zeros(2, device=self.device, dtype=torch.int64) if health else None
        d = L.RolloutVjpDesc()
        d.struct_size = C.sizeof(L.RolloutVjpDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.z0_dev, d.u_dev = z0.data_ptr(), Ut.data_ptr()
        d.u_stride_t, d.u_stride_n = st, sn
        # an empty gtraj (stride > T: no snapshot) is no trajectory term
        d.gtraj_dev = gt.data_ptr() if (gt is not None and gt.numel()) else None
        d.stride = int(stride)
        d.gzT_dev = gT.data_ptr() if gT is not None else None
        d.gz0_dev, d.gu_dev, d.z_out_dev = gz0.data_ptr(), gU.data_ptr(), z.data_ptr()
        d.workspace_dev, d.workspace_bytes = ws.data_ptr(), ws.numel() * 8
        d.health_dev = hc.data_ptr() if hc is not None else None
        d.singular_eps = float(singular_eps)
        gkp = None
        with torch.cuda.device(self.device):
            if coef:
                gkp = torch.empty((L.NKP, n), device=self.device, dtype=torch.float64)
                dc = L.RolloutVjpCoefDesc()
                dc.struct_size = C.sizeof(L.RolloutVjpCoefDesc)
                dc.vjp = d
                dc.gkp_dev = gkp.data_ptr()
                L.check(L.lib.brov_rollout_vjp_coef(self._h, C.byref(dc), self._stream()))
                gkp = gkp.t()
            else:
                L.check(L.lib.brov_rollout_vjp(self._h, C.byref(d), self._stream()))
        return VjpResult(gx0=gz0[:, :self.nx], glag0=self._glag0(gz0, lag_repr, n), gU=gU, z=z, health=hc, gkp=gkp)

    def rollout_diff(self, x0: torch.Tensor, U: torch.Tensor, lag0: Optional[torch.Tensor] = None, dt: float = 0.02,
                     integrator: str = "rk4", stride: int = 1, lag_repr: str = "projected",
                     kp: Optional[torch.Tensor] = None):
        """Differentiable rollout: (traj [T//stride, N, NX] or None for stride 0, xT [N, NX], lagT [N, 18] or None)
        as `rollout` returns them, with torch autograd gradients to x0, U [T, N, NU] (per vehicle) and lag0 [N, 18].
        The forward is `rollout`; the backward is one `rollout_vjp` call.  The lag is exchanged in projected
        coordinates (lag_repr="projected"), the form whose derivative the adjoint carries.
        kp (float64, [NKP] shared or [N, NKP] per vehicle, e.g. from derive_params_torch): the rollout runs with these
        kernel coefficients instead of the engine's, and their gradient flows back (rollout_vjp(coef=True), summed
        over the vehicles for [NKP]).  The engine's own coefficients and table are restored after the forward and
        the backward, also when either raises."""
        if lag_repr != "projected":
            raise ValueError("rollout_diff exchanges the projected lag: lag_repr must be 'projected'")
        if kp is not None:
            n = x0.shape[0]
            if not isinstance(kp, torch.Tensor) or kp.dtype != torch.float64:
                raise ValueError("kp must be a float64 tensor")
            if tuple(kp.shape) not in ((L.NKP,), (n, L.NKP)):
                raise ValueError(f"kp must have shape [{L.NKP}] or [{n}, {L.NKP}], got {tuple(kp.shape)}")
            if self.dtype != "f64" or self.is_di:
                raise ValueError("coefficient gradients need an fp64 engine of a Fossen model")
            kp = kp.to(self.device)
        lag_t = lag0 if (lag0 is not None and self.model == "thruster8") else None
        traj, xT, lagT = _RolloutDiff.apply(self, x0, U, lag_t, float(dt), integrator, int(stride), kp)
        return (traj if stride else None), xT, (lagT if self.model == "thruster8" else None)

    def _cl_operand(self, v, inner: tuple, layout: str, n: int, what: str):
        """(tensor, stride_t, stride_n, T or None) of a closed-loop operand with trailing shape `inner`"""
        t = self.tensor(v)
        nd = len(inner)
        if layout == "auto":
            extra = t.dim() - nd
            layout = {0: "const_shared", 1: "shared", 2: "tnc"}.get(extra)
            if layout is None:
                raise ValueError(f"{what} has {t.dim()} dimensions; expected {nd} to {nd + 2}")
        if layout not in _CL_LAYOUTS:
            raise ValueError(f"{what} layout must be auto|" + "|".join(_CL_LAYOUTS))
        size = int(np.prod(inner))
        lead = {"const_shared": (), "shared": (None,), "const": (n,), "tnc": (None, n)}[layout]
        if t.dim() != len(lead) + nd or tuple(t.shape[len(lead):]) != inner or \
                any(w is not None and t.shape[q] != w for q, w in enumerate(lead)):
            want = ", ".join(["T" if w is None else str(w) for w in lead] + [str(q) for q in inner])
            raise ValueError(f"{what} ({layout}) must have shape [{want}], got {tuple(t.shape)}")
        st, sn = {"const_shared": (0, 0), "shared": (size, 0), "const": (0, size), "tnc": (n * size, size)}[layout]
        T_ = t.shape[0] if layout in ("shared", "tnc") else None
        return t, st, sn, T_

    def _cl_setup(self, x0, K, z_ref, u_ref, steps, lag0, lag_repr, k_layout, ref_layout, u_min, u_max):
        """(n, steps, z0, (K, st, sn), (z_ref, st, sn), (u_ref, st, sn), u_min [NU], u_max [NU]) of a closed-loop call"""
        x0 = self.tensor(x0)
        self._check_rows(x0, self.nx, "x0")
        n = x0.shape[0]
        nz, nu = self.nz, self.nu
        Kt, kst, ksn, kT = self._cl_operand(K, (nu, nz), k_layout, n, "K")
        zr, zst, zsn, zT = self._cl_operand(z_ref, (nz,), ref_layout, n, "z_ref")
        ur, ust, usn, uT = self._cl_operand(u_ref, (nu,), ref_layout, n, "u_ref")
        Ts = {t for t in (kT, zT, uT) if t is not None}
        if steps is not None:
            Ts.add(int(steps))
        if len(Ts) != 1:
            raise ValueError("the time-varying operands disagree on T" if Ts else
                             "no operand is time-varying: give steps=")
        steps = Ts.pop()
        z0 = self._z0(x0, lag0, lag_repr, n)
        lim = 1.0 if self.model == "thruster8" else np.inf
        lo = np.broadcast_to(np.asarray(-lim if u_min is None else u_min, float), (nu,))
        hi = np.broadcast_to(np.asarray(lim if u_max is None else u_max, float), (nu,))
        return n, steps, z0, (Kt, kst, ksn), (zr, zst, zsn), (ur, ust, usn), lo, hi

    def closed_loop(self, x0, K, z_ref, u_ref, steps: Optional[int] = None, dt: float = 0.02, integrator: str = "rk4",
                    lag0=None, lag_repr: str = "thruster", k_layout: str = "auto", ref_layout: str = "auto",
                    u_min=None, u_max=None, stride: int = 0, want_u: bool = False, cost_q=None, cost_r=None,
                    cost: Optional[torch.Tensor] = None, cost_accumulate: bool = False,
                    z_out: Optional[torch.Tensor] = None, health: bool = False,
                    singular_eps: float = 0.0) -> ClosedLoopResult:
        """Closed-loop rollout of N vehicles with an affine state-feedback law evaluated in the kernel
        (brov_closed_loop): at every step k, with z_k = [x_k | Z_k] as in `linearize` (NZ = 30 / 12 / 13),
            dz = z_k - z_ref_k   (Euler-angle models: angles wrapped to (-pi, pi]),
            u_k = clamp(u_ref_k - K_k dz, u_min, u_max),   z_{k+1} = the rollout's step from z_k under u_k.

        K has rows [NU, NZ] (the K numpy builds from a DARE solution), z_ref [NZ], u_ref [NU].  Each operand has one
        of four layouts (k_layout / ref_layout; ref_layout applies to z_ref and u_ref):
          "const_shared" [...]        one value for every vehicle and step
          "shared"       [T, ...]     time-varying, shared by every vehicle
          "const"        [N, ...]     constant per vehicle (never chosen by "auto": name it)
          "tnc"          [T, N, ...]  time-varying per vehicle
        "auto" picks from the number of dimensions.  T comes from the time-varying operands, which must agree; with
        none of them give steps=.  lag0 (thruster model): per-thruster [N,24] (lag_repr="thruster") or projected
        [N,18] (lag_repr="projected"); None = zeros.  The result is always in projected lag coordinates.

        u_min / u_max: scalars or per-channel (default +-1 for thruster8, unbounded for the wrench models).
        stride > 0 returns z after every stride-th step (z_traj [T//stride, N, NZ]); want_u adds the applied inputs of
        those steps (u_traj [T//stride, N, NU]).  cost_q [NZ] / cost_r [NU] (diagonal weights) turn on the cost
        sum_k dz'Q dz + (u_k - u_ref_k)'R (u_k - u_ref_k) per vehicle, written into `cost` if given and added to its
        values with cost_accumulate (chunked calls add up bit for bit).  The engine's shared coefficients or its
        per-vehicle table (set_vehicle_physical, N rows) are used."""
        n, steps, z0, (Kt, kst, ksn), (zr, zst, zsn), (ur, ust, usn), lo, hi = self._cl_setup(
            x0, K, z_ref, u_ref, steps, lag0, lag_repr, k_layout, ref_layout, u_min, u_max)
        nz, nu = self.nz, self.nu
        if z_out is None:
            z_out = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        else:
            self._check_lag_inout(z_out, n, nz)
        zt = ut = None
        if stride:
            S = steps // int(stride)
            zt = torch.empty((S, n, nz), device=self.device, dtype=self.tdtype)
            ut = torch.empty((S, n, nu), device=self.device, dtype=self.tdtype) if want_u else None
        want_cost = cost is not None or cost_q is not None or cost_r is not None
        if want_cost:
            if cost is None:
                cost = torch.zeros(n, device=self.device, dtype=self.tdtype)
            self._check_lag_inout(cost, n, 1)
        hc = torch.zeros(2, device=self.device, dtype=torch.int64) if health else None
        d = L.ClosedLoopDesc()
        d.struct_size = C.sizeof(L.ClosedLoopDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.z0_dev, d.z_out_dev = z0.data_ptr(), z_out.data_ptr()
        d.K_dev, d.K_stride_t, d.K_stride_n = Kt.data_ptr(), kst, ksn
        d.z_ref_dev, d.z_ref_stride_t, d.z_ref_stride_n = zr.data_ptr(), zst, zsn
        d.u_ref_dev, d.u_ref_stride_t, d.u_ref_stride_n = ur.data_ptr(), ust, usn
        for r in range(nu):
            d.u_min[r], d.u_max[r] = float(lo[r]), float(hi[r])
        self._cost_weights(d, cost_q, cost_r)
        d.traj_dev = zt.data_ptr() if zt is not None and zt.numel() else None
        d.u_traj_dev = ut.data_ptr() if ut is not None and ut.numel() else None
        d.stride = int(stride)
        d.cost_dev = cost.data_ptr() if want_cost else None
        d.cost_accumulate = int(bool(cost_accumulate))
        d.health_dev = hc.data_ptr() if hc is not None else None
        d.singular_eps = float(singular_eps)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_closed_loop(self._h, C.byref(d), self._stream()))
        return ClosedLoopResult(z=z_out, z_traj=zt, u_traj=ut, cost=cost if want_cost else None, health=hc)

    def closed_loop_vjp(self, x0, K, z_ref, u_ref, gtraj=None, gzT=None, gcost=None, stride: int = 0,
                        want: Sequence[str] = ("K", "z_ref", "u_ref"), steps: Optional[int] = None, dt: float = 0.02,
                        integrator: str = "rk4", lag0=None, lag_repr: str = "thruster", k_layout: str = "auto",
                        ref_layout: str = "auto", u_min=None, u_max=None, cost_q=None, cost_r=None,
                        health: bool = False, singular_eps: float = 0.0) -> ClosedLoopVjpResult:
        """Reverse-mode gradients of N closed-loop rollouts (brov_closed_loop_vjp): for every vehicle, with the
        feedback law, layouts, bounds and cost weights of `closed_loop`,
            L = sum_{k = stride, 2 stride, ... <= T} <c_k, z_k> + <g_T, z_T> + g_c cost,
        returns dL/dz_0 (as gx0 and glag0) and, for the operands named in `want`, dL/dK, dL/dz_ref and dL/du_ref in
        the shape of the operand passed (a shared dimension gets the sum over it).  The feedback is differentiated
        through: the clamp has derivative 0 on a saturated channel, the angle wrap derivative 1; the step is
        differentiated as `rollout_vjp` differentiates it.

        gtraj [T//stride, N, NZ]: c_k on the full z, in the layout of closed_loop's z_traj (None: no trajectory term);
        gzT [N, NZ] (None: zero); gcost: g_c, a scalar or [N] (None: no cost term).  lag0 (thruster model):
        per-thruster [N,24] with lag_repr="thruster", projected [N,18] with "projected"; glag0 comes back in the same
        representation.  The call allocates the workspace the request needs (z_k, plus the cotangents of the operands in
        `want`).  fp64 engines; the engine's shared coefficients or its per-vehicle table (N rows)."""
        want = tuple(want)
        bad = set(want) - {"K", "z_ref", "u_ref"}
        if bad:
            raise ValueError(f"want names operands among K, z_ref, u_ref, not {sorted(bad)}")
        n, steps, z0, (Kt, kst, ksn), (zr, zst, zsn), (ur, ust, usn), lo, hi = self._cl_setup(
            x0, K, z_ref, u_ref, steps, lag0, lag_repr, k_layout, ref_layout, u_min, u_max)
        nz, nu = self.nz, self.nu
        gt, gT = self._cotangents(gtraj, gzT, steps, stride, n, nz)
        gc = None
        if gcost is not None:
            gc = torch.as_tensor(gcost, dtype=self.tdtype, device=self.device)
            gc = (gc.expand(n) if gc.dim() == 0 else gc.reshape(n)).contiguous()
        gz0 = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        z = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        outs = {w: torch.empty_like(t) if w in want else None for w, t in (("K", Kt), ("z_ref", zr), ("u_ref", ur))}
        # the workspace this request needs (include/brov.h): z_k and the requested operands' cotangents per vehicle and
        # step, plus one scratch row per vehicle for an operand whose strides are both 0
        per, scr = nz, 0
        for w, E, st_, sn_ in (("K", nu * nz, kst, ksn), ("z_ref", nz, zst, zsn), ("u_ref", nu, ust, usn)):
            if w in want:
                per += nz if w == "z_ref" else nu
                scr = max(scr, E) if st_ == 0 and sn_ == 0 else scr
        ws = torch.empty(max(n * (steps * per + scr), 1), device=self.device, dtype=torch.float64)
        hc = torch.zeros(2, device=self.device, dtype=torch.int64) if health else None
        d = L.ClosedLoopVjpDesc()
        d.struct_size = C.sizeof(L.ClosedLoopVjpDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.z0_dev = z0.data_ptr()
        d.K_dev, d.K_stride_t, d.K_stride_n = Kt.data_ptr(), kst, ksn
        d.z_ref_dev, d.z_ref_stride_t, d.z_ref_stride_n = zr.data_ptr(), zst, zsn
        d.u_ref_dev, d.u_ref_stride_t, d.u_ref_stride_n = ur.data_ptr(), ust, usn
        for r in range(nu):
            d.u_min[r], d.u_max[r] = float(lo[r]), float(hi[r])
        self._cost_weights(d, cost_q, cost_r)
        # an empty gtraj (stride > T: no snapshot) is no trajectory term
        d.gtraj_dev = gt.data_ptr() if (gt is not None and gt.numel()) else None
        d.stride = int(stride)
        d.gzT_dev = gT.data_ptr() if gT is not None else None
        d.gcost_dev = gc.data_ptr() if gc is not None else None
        d.gz0_dev, d.z_out_dev = gz0.data_ptr(), z.data_ptr()
        d.gK_dev = outs["K"].data_ptr() if outs["K"] is not None else None
        d.gz_ref_dev = outs["z_ref"].data_ptr() if outs["z_ref"] is not None else None
        d.gu_ref_dev = outs["u_ref"].data_ptr() if outs["u_ref"] is not None else None
        d.workspace_dev, d.workspace_bytes = ws.data_ptr(), ws.numel() * 8
        d.health_dev = hc.data_ptr() if hc is not None else None
        d.singular_eps = float(singular_eps)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_closed_loop_vjp(self._h, C.byref(d), self._stream()))
        return ClosedLoopVjpResult(gx0=gz0[:, :self.nx], glag0=self._glag0(gz0, lag_repr, n), gK=outs["K"], gz_ref=outs["z_ref"], gu_ref=outs["u_ref"],
                                   z=z, health=hc)

    def closed_loop_diff(self, x0: torch.Tensor, K: torch.Tensor, z_ref: torch.Tensor, u_ref: torch.Tensor,
                         lag0: Optional[torch.Tensor] = None, steps: Optional[int] = None, dt: float = 0.02,
                         integrator: str = "rk4", stride: int = 0, k_layout: str = "auto", ref_layout: str = "auto",
                         u_min=None, u_max=None, cost_q=None, cost_r=None):
        """Differentiable closed-loop rollout: (z_traj [T//stride, N, NZ] or None for stride 0, z [N, NZ], cost [N] or
        None without cost weights) as `closed_loop` returns them, with torch autograd gradients to x0, lag0 (projected,
        [N, 18]), K, z_ref and u_ref in any of the four operand layouts.  The forward is `closed_loop`; the backward is
        one `closed_loop_vjp` call.  The engine's shared coefficients or its per-vehicle table are used."""
        if self.dtype != "f64" or self.is_di:
            raise ValueError("closed-loop gradients need an fp64 engine of a Fossen model")
        lag_t = lag0 if (lag0 is not None and self.model == "thruster8") else None
        opts = dict(steps=steps, dt=float(dt), integrator=integrator, stride=int(stride), k_layout=k_layout,
                    ref_layout=ref_layout, u_min=u_min, u_max=u_max, cost_q=cost_q, cost_r=cost_r)
        zt, z, cost = _ClosedLoopDiff.apply(self, opts, x0, lag_t, K, z_ref, u_ref)
        want_cost = cost_q is not None or cost_r is not None
        return (zt if stride else None), z, (cost if want_cost else None)

    def ekf(self, x0, P0, U, Y, q, r, dt: float = 0.02, integrator: str = "rk4", lag0=None, lag_repr: str = "thruster",
            u_layout: str = "auto", y_layout: str = "auto", stride: int = 0, want_cov: bool = False, stats=None,
            stats_accumulate: bool = False, health: bool = False, singular_eps: float = 0.0) -> EkfResult:
        """N extended Kalman filters on the engine's model (brov_ekf), each over its own measurement series: at every
        step k the prediction x- = Phi(z_k, u_k), P- = A_k P_k A_k^T + diag(q) with the exact step Jacobian A_k of
        `linearize`, then one scalar update per component j with a finite Y[k, j] (NaN = not measured), in order:
            nu = y_j - x-_j (angles wrapped to one turn), s = P-_jj + r_j, g = P-[:, j] / s,
            x- += g nu, P- = (I - g e_j') P- (I - g e_j')' + r_j g g'  (Joseph form),
            loglik -= (nu^2 / s + log s + log 2 pi) / 2, nis += nu^2 / s, count += 1.
        Y[k] measures the state AFTER the step taken with U[k]: for a recorded series X, U pass x0 = X[0],
        U = U[:-1], Y = X[1:].  The covariance covers x only (NX = 12); the projected lag is a deterministic filter
        of the inputs.  A non-finite Y entry (NaN, and also +-inf) is not measured.  q and r are checked on the host
        before the launch, so the call synchronises the engine's stream.  fp64 engines with shared coefficients,
        thruster8 and wrench12.

        x0 [N, NX]; lag0 (thruster model): per-thruster [N,24] (lag_repr="thruster") or projected [N,18]
        (lag_repr="projected"); None = zeros.  P0: [NX, NX] (one matrix for every filter), [N, NX, NX], or the
        diagonal [NX] / [N, NX] (a 2-D [NX, NX] P0 is always a full matrix).
        U: "tnc" [T, N, NU] (the default for 3-D), "shared" [T, NU] (the default for 2-D), or "const" [N, NU].
        Y: "tnc" [T, N, NX] (the default for 3-D) or "shared" [T, NX] (the default for 2-D); T comes from Y.
        q, r: diagonal process / measurement noise variances, [NX] shared or [N, NX] per filter; q >= 0, r > 0.
        stride > 0 returns x after every stride-th step (x_traj [T//stride, N, NX]), and with want_cov P at the same
        steps (P_traj).  stats: (loglik, nis, count) tensors ([N] float64, float64, int64 on the engine's device)
        to write into; with stats_accumulate the call adds to their values, so that chunked calls (carrying z and P)
        add up bit for bit."""
        x0 = self.tensor(x0)
        self._check_rows(x0, self.nx, "x0")
        n, nx, nz, nu = x0.shape[0], self.nx, self.nz, self.nu
        Yt = self.tensor(Y)
        if y_layout == "auto":
            y_layout = "tnc" if Yt.dim() == 3 else "shared"
        if y_layout == "tnc":
            if Yt.dim() != 3 or Yt.shape[1] != n or Yt.shape[2] != nx:
                raise ValueError(f"Y must have shape [T, {n}, {nx}], got {tuple(Yt.shape)}")
            yst, ysn = n * nx, nx
        elif y_layout == "shared":
            self._check_rows(Yt, nx, "Y")
            yst, ysn = nx, 0
        else:
            raise ValueError("y_layout must be auto|tnc|shared")
        steps = Yt.shape[0]
        Ut = self.tensor(U)
        if u_layout == "auto":
            u_layout = "tnc" if Ut.dim() == 3 else "shared"
        if u_layout == "tnc":
            if Ut.dim() != 3 or Ut.shape[1] != n or Ut.shape[2] != nu:
                raise ValueError(f"U must have shape [T, {n}, {nu}], got {tuple(Ut.shape)}")
            ust, usn = n * nu, nu
        elif u_layout == "shared":
            self._check_rows(Ut, nu, "U")
            ust, usn = nu, 0
        elif u_layout == "const":
            if Ut.dim() != 2 or Ut.shape[0] != n or Ut.shape[1] != nu:
                raise ValueError(f"U must have shape [{n}, {nu}], got {tuple(Ut.shape)}")
            ust, usn = 0, nu
        else:
            raise ValueError("u_layout must be auto|tnc|shared|const")
        if u_layout != "const" and Ut.shape[0] != steps:
            raise ValueError(f"U has {Ut.shape[0]} steps and Y {steps}")

        def noise(v, what):
            t = self.tensor(v)
            if t.dim() == 1 and t.shape[0] == nx:
                return t, 0
            if t.dim() == 2 and tuple(t.shape) == (n, nx):
                return t, nx
            raise ValueError(f"{what} must have shape [{nx}] or [{n}, {nx}], got {tuple(t.shape)}")
        qt, qsn = noise(q, "q")
        rt, rsn = noise(r, "r")
        P0t = self.tensor(P0)
        if P0t.dim() == 2 and tuple(P0t.shape) == (nx, nx):
            P0t = P0t.expand(n, nx, nx)
        elif P0t.dim() == 1 and P0t.shape[0] == nx:
            P0t = torch.diag_embed(P0t.expand(n, nx))
        elif P0t.dim() == 2 and tuple(P0t.shape) == (n, nx):
            P0t = torch.diag_embed(P0t)
        elif P0t.dim() != 3 or tuple(P0t.shape) != (n, nx, nx):
            raise ValueError(f"P0 must have shape [{nx}, {nx}], [{n}, {nx}, {nx}], [{nx}] or [{n}, {nx}], "
                             f"got {tuple(P0t.shape)}")
        P0t = P0t.contiguous()
        z0 = self._z0(x0, lag0, lag_repr, n)
        if stats is None:
            if stats_accumulate:
                raise ValueError("stats_accumulate needs stats=(loglik, nis, count)")
            ll = torch.empty(n, device=self.device, dtype=torch.float64)
            ni = torch.empty(n, device=self.device, dtype=torch.float64)
            cnt = torch.empty(n, device=self.device, dtype=torch.int64)
        else:
            ll, ni, cnt = stats
            for t, dty, what in ((ll, torch.float64, "loglik"), (ni, torch.float64, "nis"), (cnt, torch.int64, "count")):
                if (not isinstance(t, torch.Tensor) or t.device != self.device or t.dtype != dty
                        or not t.is_contiguous() or tuple(t.shape) != (n,)):
                    raise ValueError(f"stats {what} must be a contiguous {dty} tensor of shape [{n}] on {self.device}")
        z = torch.empty((n, nz), device=self.device, dtype=self.tdtype)
        P = torch.empty((n, nx, nx), device=self.device, dtype=self.tdtype)
        xt = Pt = None
        if stride:
            S = steps // int(stride)
            xt = torch.empty((S, n, nx), device=self.device, dtype=self.tdtype)
            Pt = torch.empty((S, n, nx, nx), device=self.device, dtype=self.tdtype) if want_cov else None
        hc = torch.zeros(2, device=self.device, dtype=torch.int64) if health else None
        d = L.EkfDesc()
        d.struct_size = C.sizeof(L.EkfDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.z0_dev, d.P0_dev = z0.data_ptr(), P0t.data_ptr()
        d.u_dev, d.u_stride_t, d.u_stride_n = Ut.data_ptr(), ust, usn
        d.y_dev, d.y_stride_t, d.y_stride_n = Yt.data_ptr(), yst, ysn
        d.q_dev, d.q_stride_n = qt.data_ptr(), qsn
        d.r_dev, d.r_stride_n = rt.data_ptr(), rsn
        d.z_out_dev, d.P_out_dev = z.data_ptr(), P.data_ptr()
        d.x_traj_dev = xt.data_ptr() if xt is not None and xt.numel() else None
        d.P_traj_dev = Pt.data_ptr() if Pt is not None and Pt.numel() else None
        d.stride = int(stride)
        d.loglik_dev, d.nis_dev, d.count_dev = ll.data_ptr(), ni.data_ptr(), cnt.data_ptr()
        d.stats_accumulate = int(bool(stats_accumulate))
        d.health_dev = hc.data_ptr() if hc is not None else None
        d.singular_eps = float(singular_eps)
        with torch.cuda.device(self.device):
            L.check(L.lib.brov_ekf(self._h, C.byref(d), self._stream()))
        return EkfResult(z=z, P=P, x_traj=xt, P_traj=Pt, loglik=ll, nis=ni, count=cnt, health=hc)

    # ------------------------------------------------------------------ host-buffer API (end-to-end path)
    def rollout_host(self, x0: np.ndarray, U: Optional[np.ndarray] = None, dt: float = 0.02, integrator: str = "rk4",
                     lag0: Optional[np.ndarray] = None, stride: int = 0, chunk_steps: int = 0,
                     out_xT: Optional[np.ndarray] = None, out_traj: Optional[np.ndarray] = None,
                     out_lag: Optional[np.ndarray] = None, lag_repr: str = "thruster", want_lag: bool = True,
                     gen: Optional[InputGenerator] = None, steps: Optional[int] = None,
                     gen_state: Optional[np.ndarray] = None, out_gen_state: Optional[np.ndarray] = None,
                     health: Optional[np.ndarray] = None):
        """Rollout with every array in HOST memory (numpy, engine dtype, C-contiguous; pinned memory overlaps the
        copies).  Inputs stream to the device in time chunks, double buffered against the kernels.
        U [T,N,NU] or [T,NU] (shared) — or gen=InputGenerator(...), steps=T: the inputs are generated on the device
        and only x0 / lag / the AR(1) state cross PCIe.  health: uint64 [2] array receiving the counts of vehicles with
        a non-finite final state / that came near theta = +-pi/2.  Returns (xT, lag or None, traj or None)."""
        def host(a, what):
            if not isinstance(a, np.ndarray) or a.dtype != self.ndtype or not a.flags.c_contiguous:
                raise ValueError(f"{what} must be a C-contiguous numpy array of dtype {np.dtype(self.ndtype)}")
            return a
        x0 = host(x0, "x0")
        n = x0.shape[0]
        if x0.shape != (n, self.nx):
            raise ValueError(f"x0 must be [N, {self.nx}]")
        if gen is not None:
            if steps is None:
                raise ValueError("generated inputs need steps=")
            steps, shared = int(steps), False
        else:
            U = host(U, "U")
            shared = U.ndim == 2
            if (shared and U.shape[1] != self.nu) or (not shared and U.shape[1:] != (n, self.nu)):
                raise ValueError("U must be [T, N, NU] or [T, NU]")
            steps = U.shape[0]
        xT = out_xT if out_xT is not None else np.empty_like(x0)
        proj = lag_repr == "projected" and self.model == "thruster8"
        nlag = 18 if proj else self.nlag
        lag_out = None
        if nlag and want_lag:
            lag_out = out_lag if out_lag is not None else np.empty((n, nlag), dtype=self.ndtype)
        traj = None
        if stride:
            traj = out_traj if out_traj is not None else np.empty((steps // stride, n, self.nx), dtype=self.ndtype)
        d = L.RolloutHostDesc()
        d.struct_size = C.sizeof(L.RolloutHostDesc)
        d.integrator = INTEGRATORS[integrator]
        d.n, d.steps, d.dt = n, steps, float(dt)
        d.x0_host, d.xT_host = x0.ctypes.data, host(xT, "out_xT").ctypes.data
        d.u_host = U.ctypes.data if gen is None else None
        d.u_shared = int(shared)
        d.lag_in_host = host(lag0, "lag0").ctypes.data if (nlag and lag0 is not None) else None
        d.lag_out_host = lag_out.ctypes.data if lag_out is not None else None
        d.traj_host = host(traj, "out_traj").ctypes.data if traj is not None else None
        d.stride = max(int(stride), 1)
        d.chunk_steps = int(chunk_steps)
        d.lag_in_repr = d.lag_out_repr = L.LAG_PROJECTED if proj else L.LAG_THRUSTER
        if gen is not None:
            gen.fill(d.gen, self.nu, host(gen_state, "gen_state").ctypes.data if gen_state is not None else None,
                     host(out_gen_state, "out_gen_state").ctypes.data if out_gen_state is not None else None)
        if health is not None:
            if health.dtype != np.uint64 or health.size < 2 or not health.flags.c_contiguous:
                raise ValueError("health must be a C-contiguous uint64 array with 2 elements")
            d.health_host = health.ctypes.data_as(C.POINTER(C.c_ulonglong))
        L.check(L.lib.brov_rollout_host(self._h, C.byref(d)))
        return xT, lag_out, traj


class _RolloutDiff(torch.autograd.Function):
    """Engine.rollout forward, Engine.rollout_vjp backward (Engine.rollout_diff)."""

    @staticmethod
    def forward(ctx, eng, x0, U, lag0, dt, integrator, stride, kp=None):
        if U.dim() != 3:
            raise ValueError("rollout_diff takes a per-vehicle U [T, N, NU]")
        thr = eng.model == "thruster8"
        with eng._coefficients(kp) if kp is not None else _nullcontext():
            r = eng.rollout(x0.detach(), U.detach(), dt=dt, integrator=integrator,
                            lag0=lag0.detach() if lag0 is not None else None, stride=stride,
                            lag_repr="projected", want_lag=thr)
        ctx.eng, ctx.dt, ctx.integrator, ctx.stride = eng, dt, integrator, stride
        ctx.has_lag = lag0 is not None
        ctx.kp = kp.detach() if kp is not None else None
        ctx.save_for_backward(x0, U, *([lag0] if lag0 is not None else []))
        n = x0.shape[0]
        traj = r.traj if stride else torch.empty((0, n, eng.nx), device=eng.device, dtype=eng.tdtype)
        lagT = r.lag if thr else torch.empty((n, 0), device=eng.device, dtype=eng.tdtype)
        return traj, r.xT, lagT

    @staticmethod
    def backward(ctx, gtraj, gxT, glagT):
        eng = ctx.eng
        saved = ctx.saved_tensors
        x0, U = saved[0], saved[1]
        lag0 = saved[2] if ctx.has_lag else None
        n = x0.shape[0]
        thr = eng.model == "thruster8"
        gx = gxT if gxT is not None else torch.zeros((n, eng.nx), device=eng.device, dtype=eng.tdtype)
        if thr:
            gl = glagT if glagT is not None else torch.zeros((n, 18), device=eng.device, dtype=eng.tdtype)
            gzT = torch.cat([gx, gl], dim=1).contiguous()
        else:
            gzT = gx.contiguous()
        gt = gtraj.contiguous() if (gtraj is not None and ctx.stride and gtraj.numel()) else None
        kp = ctx.kp
        with eng._coefficients(kp) if kp is not None else _nullcontext():
            res = eng.rollout_vjp(x0.detach(), U.detach(), gtraj=gt, gzT=gzT,
                                  stride=ctx.stride if gt is not None else 0, dt=ctx.dt, integrator=ctx.integrator,
                                  lag0=lag0.detach() if lag0 is not None else None, lag_repr="projected",
                                  u_layout="tnc", coef=kp is not None)
        glag = res.glag0 if (thr and ctx.has_lag) else None
        gkp = None
        if kp is not None:
            gkp = res.gkp.sum(0) if kp.dim() == 1 else res.gkp
        return None, res.gx0, res.gU, glag, None, None, None, gkp


class _ClosedLoopDiff(torch.autograd.Function):
    """Engine.closed_loop forward, Engine.closed_loop_vjp backward (Engine.closed_loop_diff)."""

    @staticmethod
    def forward(ctx, eng, opts, x0, lag0, K, z_ref, u_ref):
        o = dict(opts)
        r = eng.closed_loop(x0.detach(), K.detach(), z_ref.detach(), u_ref.detach(),
                            lag0=lag0.detach() if lag0 is not None else None, lag_repr="projected", **o)
        ctx.eng, ctx.opts = eng, o
        ctx.has_lag = lag0 is not None
        ctx.save_for_backward(x0, K, z_ref, u_ref, *([lag0] if lag0 is not None else []))
        n = x0.shape[0]
        zt = r.z_traj if r.z_traj is not None else torch.empty((0, n, eng.nz), device=eng.device, dtype=eng.tdtype)
        cost = r.cost if r.cost is not None else torch.empty((0,), device=eng.device, dtype=eng.tdtype)
        return zt, r.z, cost

    @staticmethod
    def backward(ctx, gzt, gz, gcost):
        eng, o = ctx.eng, dict(ctx.opts)
        saved = ctx.saved_tensors
        x0, K, z_ref, u_ref = saved[:4]
        lag0 = saved[4] if ctx.has_lag else None
        stride = o.pop("stride")
        gt = gzt.contiguous() if (gzt is not None and stride and gzt.numel()) else None
        gc = gcost.contiguous() if (gcost is not None and gcost.numel()) else None
        gT = gz.contiguous() if gz is not None else None
        need = ctx.needs_input_grad
        want = tuple(w for w, i in (("K", 4), ("z_ref", 5), ("u_ref", 6)) if need[i])
        res = eng.closed_loop_vjp(x0.detach(), K.detach(), z_ref.detach(), u_ref.detach(), gtraj=gt, gzT=gT, gcost=gc,
                                  stride=stride if gt is not None else 0, want=want,
                                  lag0=lag0.detach() if lag0 is not None else None, lag_repr="projected", **o)
        glag = res.glag0 if ctx.has_lag else None
        return None, None, res.gx0, glag, res.gK, res.gz_ref, res.gu_ref


def reduced9_rhs(x: torch.Tensor, u: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """bluerov_compute RHS on CUDA tensors x [B,9], u [B,4] (float32 or float64); `out` [B,9] is reused if given."""
    if x.dtype not in (torch.float32, torch.float64) or u.dtype != x.dtype:
        raise TypeError("x and u must both be float32 or both float64")
    if not x.is_cuda or not u.is_cuda:
        raise RuntimeError("reduced9_rhs expects CUDA tensors")
    x = x.contiguous()
    u = u.contiguous()
    if out is None:
        out = torch.empty_like(x)
    elif out.shape != x.shape or out.dtype != x.dtype or out.device != x.device or not out.is_contiguous():
        raise ValueError("out must be a contiguous tensor like x")
    with torch.cuda.device(x.device):
        L.check(L.lib.brov_reduced9_rhs(L.F32 if x.dtype == torch.float32 else L.F64, x.data_ptr(), u.data_ptr(),
                                        out.data_ptr(), x.shape[0], torch.cuda.current_stream(x.device).cuda_stream))
    return out


def fma_peak(dtype: str = "f32", device: int = 0, iters: int = 4096):
    """(TFLOP/s, ms) of an FMA-chain microbenchmark: the measured FP pipe peak of this GPU."""
    tf, ms = C.c_double(), C.c_double()
    L.check(L.lib.brov_fma_peak(DTYPES[dtype][0], int(device), int(iters), C.byref(tf), C.byref(ms)))
    return tf.value, ms.value


def pinned_empty(shape, dtype) -> np.ndarray:
    """Pinned (page-locked) host numpy array, via torch's allocator."""
    tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}[np.dtype(dtype)]
    t = torch.empty(tuple(shape), dtype=tdt, pin_memory=True)
    return t.numpy()
