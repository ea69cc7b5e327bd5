"""Numpy restatement of the extended Kalman filter of brov_ekf (include/brov.h), over a batch of N filters.

The filter is generic in the model: `step(x, aux, u) -> (x', aux')` takes one step of N filters (aux: whatever else
the step carries, e.g. the thruster lag) and `jac(x, aux, u) -> A [N, NX, NX]` is dx'/dx at the same point.  The
measurement model is a selection of state components (NaN = not measured) with diagonal R, updated one component at
a time in index order, in Joseph form; innovations of the components in `wrap` are wrapped to one turn."""
import numpy as np

LOG_2PI = float(np.log(2.0 * np.pi))


def _sym_upper(P):
    """the upper triangle of P mirrored (the kernel computes one triangle and mirrors it)"""
    return np.triu(P) + np.swapaxes(np.triu(P, 1), -1, -2)


def ekf(step, jac, x0, aux0, P0, U, Y, q, r, wrap=(3, 4, 5)):
    """x0 [N, NX], P0 [N, NX, NX], U [T, N, NU], Y [T, N, NX], q / r [NX] or [N, NX].
    Returns dict(x [N, NX], aux, P [N, NX, NX], x_traj [T, N, NX], P_traj [T, N, NX, NX], loglik [N], nis [N],
    count [N])."""
    x = np.array(x0, float)
    N, nx = x.shape
    aux = aux0
    P = np.array(P0, float).copy()
    Q = np.broadcast_to(np.asarray(q, float), (N, nx))
    R = np.broadcast_to(np.asarray(r, float), (N, nx))
    Y = np.asarray(Y, float)
    ll, nis, cnt = np.zeros(N), np.zeros(N), np.zeros(N, np.int64)
    xs, Ps = [], []
    rows = np.arange(N)
    for k in range(Y.shape[0]):
        A = jac(x, aux, U[k])
        x, aux = step(x, aux, U[k])
        x = np.array(x, float)
        P = _sym_upper(A @ P @ np.swapaxes(A, -1, -2))
        P[:, np.arange(nx), np.arange(nx)] += Q
        for j in range(nx):
            m = np.isfinite(Y[k, :, j])
            if not m.any():
                continue
            i = rows[m]
            nu = Y[k, i, j] - x[i, j]
            if j in wrap:
                nu = nu - 2.0 * np.pi * np.rint(nu / (2.0 * np.pi))
            Pi = P[i]
            s = Pi[:, j, j] + R[i, j]
            g = Pi[:, :, j] / s[:, None]
            x[i] += g * nu[:, None]
            Kf = np.eye(nx)[None] - g[:, :, None] * np.eye(nx)[j][None, None, :]      # I - g e_j^T
            Pn = Kf @ Pi @ np.swapaxes(Kf, -1, -2) + R[i, j][:, None, None] * g[:, :, None] * g[:, None, :]
            P[i] = _sym_upper(Pn)
            e2 = nu * nu / s
            ll[i] -= 0.5 * (e2 + np.log(s) + LOG_2PI)
            nis[i] += e2
            cnt[i] += 1
        xs.append(x.copy())
        Ps.append(P.copy())
    return dict(x=x, aux=aux, P=P, x_traj=np.array(xs).reshape(-1, N, nx), P_traj=np.array(Ps).reshape(-1, N, nx, nx),
                loglik=ll, nis=nis, count=cnt)


def fossen_step_jac(model, integ, h=1e-5):
    """(step, jac) on oracle/fossen_np.py for ekf(): aux is the per-thruster lag [N, 8, 3] (None for the wrench
    models); jac is the central difference of the step in x, the lag held."""
    from . import fossen_np as O

    def step(x, lag, u):
        return O.step(model, integ, x, u, lag)

    def jac(x, lag, u):
        N, nx = x.shape
        hs = h * np.maximum(1.0, np.abs(x))                                          # [N, nx]
        X = np.repeat(x[:, None, :], 2 * nx, axis=1)                                 # [N, 2nx, nx]
        idx = np.arange(nx)
        X[:, 2 * idx, idx] += hs
        X[:, 2 * idx + 1, idx] -= hs
        lagr = None if lag is None else np.repeat(lag, 2 * nx, axis=0)
        out, _ = O.step(model, integ, X.reshape(-1, nx), np.repeat(u, 2 * nx, axis=0), lagr)
        out = out.reshape(N, nx, 2, nx)
        return np.swapaxes((out[:, :, 0] - out[:, :, 1]) / (2 * hs[:, :, None]), 1, 2)
    return step, jac
