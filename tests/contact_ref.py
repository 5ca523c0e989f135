"""Independent reference of the contact plant (wbc_plant_contact_step), test infrastructure only.

It shares no source with the kernel (wbc_contact.cuh): the dynamics are the CPU oracle's dense formulation (oracle_py.update_only:
18 x 18 M, h, the stacked linear foot Jacobians), G = J M^-1 J' is formed densely, and each contact QP
    min 1/2 l'(G + eps diag(G)) l + l'(J nu_free - b)   s.t. the friction pyramid of every candidate foot
is solved by a PRIMAL active-set method on the dense KKT system (the kernel runs a dual Goldfarb-Idnani method on a Cholesky
factor).  Every QP result is certified -- stationarity, primal and dual feasibility, complementarity -- before it is used; a result
that fails certification raises instead of serving as a reference.
"""
import numpy as np

from wbc_quadruped_dob_b200 import scenarios as S

CERT_TOL = 1e-11
_ZERO_FIELDS = {"com_des_pos": 6, "com_des_vel": 6, "com_des_acc": 6, "sw_des_pos": 6, "sw_des_vel": 6, "sw_des_acc": 6,
                "foot_force": 12, "obs_yd": 6, "obs_yw": 6}


class CertificationError(AssertionError):
    pass


def pyramid_rows(mu):
    """The 5 rows of one foot's pyramid in 'a . l >= 0' form, unit length: normal, then -+x, -+y (the kernel's row order)."""
    s = 1.0 / np.sqrt(1.0 + mu * mu)
    return np.array([[0.0, 0.0, 1.0], [-s, 0.0, mu * s], [s, 0.0, mu * s], [0.0, -s, mu * s], [0.0, s, mu * s]])


def primal_active_set(H, g, A, max_iter=500):
    """min 1/2 x'Hx + g'x s.t. A x >= 0 (H positive definite), from the feasible x = 0 with an empty working set.
    Returns (x, working set, multipliers), certified."""
    nv, nr = H.shape[0], A.shape[0]
    x = np.zeros(nv)
    W = []
    scale = max(np.abs(np.linalg.solve(H, g)).max(), 1e-300)
    for _ in range(max_iter):
        Aw = A[W]
        K = np.block([[H, -Aw.T], [Aw, np.zeros((len(W), len(W)))]])
        sol = np.linalg.solve(K, np.concatenate([-(H @ x + g), np.zeros(len(W))]))
        p, lam = sol[:nv], sol[nv:]
        if np.abs(p).max() <= 1e-14 * scale:
            # multipliers at x: H x + g = Aw' mu
            mu = np.linalg.lstsq(Aw.T, H @ x + g, rcond=None)[0] if W else np.zeros(0)
            if len(W) == 0 or mu.min() >= 0.0:
                certify(H, g, A, x, W, mu)
                return x, list(W), mu
            W.pop(int(np.argmin(mu)))
            continue
        alpha, block = 1.0, -1
        ap = A @ p
        for i in range(nr):
            # a row that depends on the working set has a . p = 0 in exact arithmetic: it never blocks
            if i in W or ap[i] >= -1e-12 * np.abs(p).max() or np.linalg.matrix_rank(A[W + [i]], tol=1e-9) <= len(W):
                continue
            a = max(0.0, A[i] @ x) / -ap[i]
            if a < alpha:
                alpha, block = a, i
        x = x + alpha * p
        if block >= 0:
            W.append(block)
    raise CertificationError("primal active set: no convergence in %d iterations" % max_iter)


def kkt_residual(H, g, A, x, W, mu):
    grad = H @ x + g
    gs = max(np.abs(grad - g).max(), np.abs(g).max(), 1e-300)
    xs = max(np.abs(x).max(), np.abs(np.linalg.solve(H, g)).max(), 1e-300)
    st = np.abs(grad - (A[W].T @ mu if W else 0.0)).max() / gs
    s = A @ x
    pv = max(0.0, -s.min()) / xs
    dv = max(0.0, -mu.min()) / gs if len(mu) else 0.0
    cp = max(np.abs(mu * s[W]).max() / (gs * xs), 0.0) if len(mu) else 0.0
    return max(st, pv, dv, cp)


def certify(H, g, A, x, W, mu):
    r = kkt_residual(H, g, A, x, W, mu)
    if not r <= CERT_TOL:
        raise CertificationError("contact QP result fails the KKT certificate: scaled residual %.3e" % r)


def _rodrigues(w, th):
    k = w / np.linalg.norm(w)
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1.0 - np.cos(th)) * (Kx @ Kx)


def contact_step(oracle, st, tau, push, ground_z, mu, nsub, beta=0.2, eps=1e-8, margin=2e-3, obs_dt=0.0025):
    """One control period of every instance.  st: dict of SoA state arrays (base_pos, base_rot, base_rpy, base_vel, q, dq);
    tau [12, n], push [6, n], ground_z [4, n], mu [n].  Returns (next state dict incl. foot_force, contact flags int [4, n],
    impulses of the last step [12, n] (world axes, 0 off contact))."""
    n = st["q"].shape[1]
    dt = obs_dt / nsub
    out = {k: np.array(st[k], dtype=np.float64) for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
    out["foot_force"] = np.zeros((12, n))
    flags = np.zeros((4, n), dtype=np.int32)
    lam_out = np.zeros((12, n))
    for i in range(n):
        cur = {k: out[k][:, i:i + 1].copy() for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
        cur.update({k: np.zeros((m, 1)) for k, m in _ZERO_FIELDS.items()})
        cur["mode"] = np.zeros(1, dtype=np.int32)
        for _ in range(nsub):
            d = oracle.update_only(cur, 0)
            M = np.array(d.M).reshape(18, 18)
            h = np.array(d.h)
            Jall = np.array(d.Jac_lin).reshape(12, 18)
            fp = np.array(d.foot_pos).reshape(4, 3)
            fR = np.array(d.foot_R).reshape(4, 3, 3)
            nu = np.concatenate([cur["base_vel"][:, 0], cur["dq"][:, 0]])
            xbc = np.array(d.com) - cur["base_pos"][:, 0]
            b = -h.copy()
            b[:3] += push[:3, i]
            b[3:6] += push[3:, i] + np.cross(xbc, push[:3, i])
            b[6:] += tau[:, i]
            nu = nu + dt * np.linalg.solve(M, b)
            phi = fp[:, 2] - ground_z[:, i]
            cand = [k for k in range(4) if phi[k] <= margin]
            lam = np.zeros(12)
            fl = np.zeros(4, dtype=np.int32)
            if cand:
                J = np.vstack([Jall[3 * k:3 * k + 3] for k in cand])
                X = np.linalg.solve(M, J.T)
                G = J @ X
                H = G + eps * np.diag(np.diag(G))
                g = J @ nu
                for f, k in enumerate(cand):
                    g[3 * f + 2] += (1.0 if phi[k] >= 0.0 else beta) * phi[k] / dt
                A = np.zeros((5 * len(cand), 3 * len(cand)))
                for f in range(len(cand)):
                    A[5 * f:5 * f + 5, 3 * f:3 * f + 3] = pyramid_rows(mu[i])
                x, W, _ = primal_active_set(H, g, A)
                for f, k in enumerate(cand):
                    rows = {r - 5 * f for r in W if 5 * f <= r < 5 * f + 5}
                    lk = x[3 * f:3 * f + 3].copy()
                    if 0 in rows or (mu[i] > 0.0 and ({1, 2} <= rows or {3, 4} <= rows)) or lk[2] <= 0.0:
                        lk[:] = 0.0
                    x[3 * f:3 * f + 3] = lk
                    fl[k] = 0 if lk[2] <= 0.0 else (2 if rows - {0} else 1)
                    lam[3 * k:3 * k + 3] = lk
                nu = nu + X @ x
            # semi-implicit Euler, exponential map of the base rotation
            cur["base_vel"][:, 0] = nu[:6]
            cur["dq"][:, 0] = nu[6:]
            cur["q"][:, 0] += dt * nu[6:]
            cur["base_pos"][:, 0] += dt * nu[:3]
            R = cur["base_rot"][:, 0].reshape(3, 3)
            wn = np.linalg.norm(nu[3:6])
            if wn > 0.0:
                R = _rodrigues(nu[3:6], wn * dt) @ R
            cur["base_rot"][:, 0] = R.reshape(9)
            cur["base_rpy"][:, 0] = [np.arctan2(R[2, 1], R[2, 2]), np.arctan2(-R[2, 0], np.hypot(R[2, 1], R[2, 2])), np.arctan2(R[1, 0], R[0, 0])]
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq"):
            out[k][:, i] = cur[k][:, 0]
        for k in range(4):
            out["foot_force"][3 * k:3 * k + 3, i] = fR[k].T @ lam[3 * k:3 * k + 3] / dt
        flags[:, i] = fl
        lam_out[:, i] = lam
    return out, flags, lam_out


def foot_heights(st):
    """World z of the four foot points, [4, n] (stacked order)."""
    _, feet = S.forward_kinematics(st["base_pos"], st["base_rot"], st["q"])
    return feet[:, :, 2].T.copy()
