"""Host side of the B200 engine: torch provides device memory and streams, libbrov.so (C ABI) does the work.

`Engine` is the batched counterpart of the reference's model objects: where the reference evaluates one vehicle per
Python call (`rov.dynamics`, `simulate_physics`, `multistep_rmse_endpoint_physics`), an Engine call covers N
vehicles / windows with one kernel launch.  Array conventions follow the reference: a state is a row
`[x y z phi theta psi u v w p q r]` (or the 13-state quaternion row), an input row is 8 thruster voltages or a
6-component body wrench.
"""
from __future__ import annotations

import ctypes as C
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
        L.check(L.lib.brov_set_vehicle_params(self._h, soa.data_ptr(), soa.shape[1], int(any_current)))

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
