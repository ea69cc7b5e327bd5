"""Multi-GPU plumbing: one process per GPU, `torch.distributed` (NCCL on B200s, gloo in CPU tests).

The path shards without any data-path exchange: vehicles of a rollout, windows of the RMSE evaluator and candidates
of an evaluator sweep are independent, so each rank takes a contiguous index range.  The only collective is the sum of
the per-rank squared error vectors and health counters (6 doubles) of the evaluator, or of the [P, 4] table of a
sweep."""
from __future__ import annotations

import os
from typing import Callable, Sequence

import numpy as np
import torch
import torch.distributed as dist


def init_from_env(backend: str = None) -> tuple[int, int, int]:
    """(rank, world, local_rank) from torchrun's environment; initialises the default group when world > 1."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return rank, world, local


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block partition of range(n): [lo, hi) of `rank`; sizes differ by at most one."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def window_shard(T: int, horizons: Sequence[int], rank: int, world: int):
    """Rows and windows of one rank for the sliding-window evaluator.
    Global windows k = 0..T-Hmin-1 are block-partitioned; the rank needs series rows [lo, min(T, hi + Hmax)) — an
    Hmax-row halo replicated at load time, no exchange.  Returns (row_lo, row_hi, n_windows_local)."""
    hmin, hmax = min(horizons), max(horizons)
    nwin = max(T - hmin, 0)
    lo, hi = shard_range(nwin, rank, world)
    return lo, min(T, hi + hmax) if hi > lo else lo, hi - lo


def window_shard_carry(T: int, H: int, rank: int, world: int, carry_steps: int):
    """Shard of the carried-lag evaluator (one horizon): besides the H-row halo after its last window a rank needs the
    input rows its first window replays — the last `carry_steps` lag steps of the shared model object's history, i.e.
    rows back to window (lo * H - carry_steps) // H.  Returns (row_lo, row_hi, n_windows_local, window_lo)."""
    nwin = max(T - H, 0)
    lo, hi = shard_range(nwin, rank, world)
    if hi <= lo:
        return lo, lo, 0, lo
    row_lo = max(0, (lo * H - int(carry_steps)) // H)
    return row_lo, min(T, hi + H), hi - lo, lo


def sharded_multistep_rmse_carry(engine, X: np.ndarray, U: np.ndarray, H: int, dt: float, integrator: str, rank: int,
                                 world: int) -> float:
    """The reference's literal evaluator semantics (lag state carried from window to window) on `world` GPUs: each
    rank scores a contiguous block of windows and replays the tail of the shared history from its own copy of the
    input rows; one all-reduce of the squared-error sum.  `engine`: a thruster-model Engine on the rank's device."""
    T = len(X)
    depth = engine.carry_steps(dt, integrator)
    row_lo, row_hi, nloc, win_lo = window_shard_carry(T, int(H), rank, world, depth)
    vec = torch.zeros(1, dtype=torch.float64, device=engine.device)
    if nloc > 0:
        se, _ = engine.multistep_se(X[row_lo:row_hi], U[row_lo:row_hi], [int(H)], dt=dt, integrator=integrator,
                                    n_windows=nloc, lag_mode="carry", window0=win_lo, row0=row_lo)
        vec += se[:1]
    allreduce_sum_(vec)
    cnt = max(T - int(H), 0)
    return float(np.sqrt(vec.item() / (cnt * X.shape[1]))) if cnt > 0 else float("nan")


class ShardedEvaluator:
    """Multi-step endpoint squared error of ONE recorded series on `world` GPUs, as a replayable step.

    Each rank owns a contiguous block of windows (plus the halo rows they read); one evaluation is
    `se_kernel -> se_finish_kernel -> all-reduce` of a 6-double vector [se_H0..se_H3, n_nonfinite, n_near_singular]
    (lag_mode="carry": one se_kernel pass per horizon, concurrent on forked streams, ONE all-reduce).
    The whole chain is captured ONCE in a CUDA graph (the NCCL all-reduce included) and replayed: at 125,000 windows per
    GPU the kernels take ~0.85 ms, so the ~0.2 ms of per-call host work (descriptor packing, three launches, a clone
    and an eager all-reduce) of the round-1 loop was a fifth of the step.  `use_graph=False` keeps the eager chain
    (gloo / CPU tests, or a torch build that cannot capture the collective)."""

    def __init__(self, engine, X, U, horizons: Sequence[int], dt: float = 0.02, integrator: str = "rk4", rank: int = 0,
                 world: int = 1, lag_mode: str = "reset", use_graph: bool = True, singular_eps: float = 0.0):
        self.e, self.hs = engine, [int(h) for h in horizons]
        self.dt, self.integ, self.lag_mode, self.world = float(dt), integrator, lag_mode, world
        self.eps = float(singular_eps)
        T = len(X)
        self.T, self.nx = T, X.shape[1]
        self.carry = lag_mode == "carry" and engine.model == "thruster8"
        dev = engine.device
        from . import _lib as L
        # passes: (horizons, first local row, n_rows, n_windows, window0, row0).  reset: ONE pass scores every horizon
        # (H = 1 and 10 are prefixes of the H = 100 rollout).  carry: the lag history a window inherits depends on the
        # horizon (the reference runs one evaluation per horizon on one shared model object), so one pass per horizon
        # — launched longest first on separate streams inside the same graph, so that the short passes fill the tail
        # of the long one instead of each paying its own partial last wave.
        if self.carry:
            depth = engine.carry_steps(dt, integrator)
            shards = [window_shard_carry(T, h, rank, world, depth) for h in self.hs]
            lo = min((s[0] for s in shards if s[2] > 0), default=0)
            hi = max((s[1] for s in shards if s[2] > 0), default=0)
            self.passes = [([h], s[0] - lo, s[1] - s[0], s[2], s[3], s[0]) for h, s in zip(self.hs, shards)]
            self.passes.sort(key=lambda p: -p[0][0])
        else:
            lo, hi, nloc = window_shard(T, self.hs, rank, world)
            self.passes = [(self.hs, 0, hi - lo, nloc, 0, 0)]
        self.nloc = sum(p[3] for p in self.passes)
        self.X = engine.tensor(X[lo:hi]).contiguous()
        self.U = engine.tensor(U[lo:hi]).contiguous()
        self.buf = torch.zeros(8, dtype=torch.float64, device=dev)      # [se x4, health x2, pad x2]
        npass = len(self.passes)
        self.se = torch.zeros((npass, 8), dtype=torch.float64, device=dev)
        self.hc = torch.zeros((npass, 2), dtype=torch.int64, device=dev)
        self.ws = [torch.empty(int(L.lib.brov_se_workspace_bytes(max(p[3], 1))), dtype=torch.uint8, device=dev)
                   for p in self.passes]
        self.side = [torch.cuda.Stream(device=dev) for _ in range(npass - 1)]
        self.graph = None
        self._eager()                      # warm-up: initialises NCCL for this size
        torch.cuda.synchronize(dev)
        if use_graph:
            try:
                g = torch.cuda.CUDAGraph()
                s = torch.cuda.Stream(device=dev)
                s.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(s):
                    self._eager()
                torch.cuda.current_stream(dev).wait_stream(s)
                torch.cuda.synchronize(dev)
                with torch.cuda.graph(g, stream=s):
                    self._eager()
                self.graph = g
            except Exception as ex:        # capture of the collective not supported by this torch / NCCL pairing
                self.graph = None
                self.capture_error = repr(ex)
                torch.cuda.synchronize(dev)

    def _pass(self, i):
        hs, r0, nrows, nwin, win0, row0 = self.passes[i]
        if nwin > 0:
            self.e.multistep_se(self.X[r0:r0 + nrows], self.U[r0:r0 + nrows], hs, dt=self.dt, integrator=self.integ,
                                n_windows=nwin, lag_mode=self.lag_mode, window0=win0, row0=row0, se_out=self.se[i],
                                health_out=self.hc[i], singular_eps=self.eps, workspace=self.ws[i])
        else:
            self.se[i].zero_()
            self.hc[i].zero_()

    def _eager(self):
        cur = torch.cuda.current_stream(self.e.device)
        self._pass(0)
        for i, s in enumerate(self.side, start=1):      # fork: the other passes on their own streams
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                self._pass(i)
        for s in self.side:                              # join
            cur.wait_stream(s)
        if self.carry:
            for i, p in enumerate(self.passes):
                self.buf[self.hs.index(p[0][0])] = self.se[i, 0]
        else:
            self.buf[:4] = self.se[0, :4]
        self.buf[4:6] = self.hc.sum(dim=0).to(torch.float64)
        allreduce_sum_(self.buf)

    def run(self) -> torch.Tensor:
        """One evaluation; returns the reduced device vector (valid after the stream has run it)."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._eager()
        return self.buf

    def rmse(self):
        """(rmse per horizon, [n_nonfinite, n_near_singular]) of the last run."""
        v = self.buf.cpu().numpy()
        cnt = global_counts(self.T, self.hs)
        r = [float(np.sqrt(v[i] / (cnt[i] * self.nx))) if cnt[i] > 0 else float("nan") for i in range(len(self.hs))]
        return r, [int(round(v[4])), int(round(v[5]))]


def allreduce_sum_(t: torch.Tensor) -> torch.Tensor:
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def global_counts(T: int, horizons: Sequence[int]) -> list[int]:
    return [max(T - int(h), 0) for h in horizons]


def sharded_sweep(local_fn: Callable[[int, int], torch.Tensor], P: int, rank: int, world: int,
                  width: int = 4) -> torch.Tensor:
    """Candidate sweep on `world` GPUs: candidates [lo, hi) of `rank` (shard_range) are scored on the whole series by
    local_fn(lo, hi) -> [hi - lo, width] squared-error sums (on the GPU: Engine.multistep_se_sweep on the rank's rows of
    the table; in CPU tests a stand-in) and written into the rank's slice of a zero [P, width] float64 tensor; one
    all-reduce assembles the table.  Exact: every entry is one rank's value plus zeros.  width = BROV_MAX_H."""
    lo, hi = shard_range(int(P), rank, world)
    part = local_fn(lo, hi) if hi > lo else None
    dev = part.device if part is not None else (torch.device("cuda", torch.cuda.current_device())
                                                if dist.is_initialized() and dist.get_backend() == "nccl" else torch.device("cpu"))
    out = torch.zeros((int(P), width), dtype=torch.float64, device=dev)
    if part is not None:
        out[lo:hi] = part.to(torch.float64)
    return allreduce_sum_(out)


def sharded_multistep_rmse(local_se: Callable[[np.ndarray, np.ndarray, Sequence[int], int], torch.Tensor],
                           X: np.ndarray, U: np.ndarray, horizons: Sequence[int], rank: int, world: int):
    """Endpoint RMSE per horizon of the whole series, computed by `world` ranks.

    local_se(X_rows, U_rows, horizons, n_windows) -> tensor of per-horizon squared-error sums for the rank's
    windows (on the GPU: Engine.multistep_se; in CPU tests: the oracle).  The sums are all-reduced, then
    rmse_h = sqrt(se_h / ((T - H_h) * n_states))."""
    T = len(X)
    hs = [int(h) for h in horizons]
    lo, hi, nloc = window_shard(T, hs, rank, world)
    if nloc > 0:
        se = local_se(X[lo:hi], U[lo:hi], hs, nloc)
    else:
        se = None
    dev = se.device if se is not None else (torch.device("cuda", torch.cuda.current_device())
                                            if dist.is_initialized() and dist.get_backend() == "nccl" else torch.device("cpu"))
    vec = torch.zeros(len(hs), dtype=torch.float64, device=dev)
    if se is not None:
        vec += se[:len(hs)].to(torch.float64)
    allreduce_sum_(vec)
    cnt = global_counts(T, hs)
    vals = vec.cpu().numpy()
    nx = X.shape[1]
    return [float(np.sqrt(vals[i] / (cnt[i] * nx))) if cnt[i] > 0 else float("nan") for i in range(len(hs))]
