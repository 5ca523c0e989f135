"""Independent reference of the contact plant's terrain form (wbc_plant_contact_step_terrain), test infrastructure only.

Like tests/contact_ref.py, whose certified primal active-set QP (primal_active_set) and pyramid rows it uses, it shares no source
with the kernel: the dynamics are the CPU oracle's dense formulation (oracle_py.update_only), G = J M^-1 J' is formed densely.
Foot k stands on the plane n_k . p = d_k with the frame F_k = [t1 t2 n] and mu_k of the terrain layout [40][n] (rows 10k..10k+2 n,
+3..+5 t1, +6..+8 t2, +9 mu): its gap is n_k . p_k - d_k, its Jacobian rows are F_k' J, and its pyramid uses its own mu.
"""
import numpy as np

from tests.contact_ref import _ZERO_FIELDS, _rodrigues, primal_active_set, pyramid_rows

STATE = ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")


def frame(terrain, k, i):
    """F = [t1 t2 n] of foot k of instance i, 3 x 3 (columns)."""
    return np.column_stack([terrain[10 * k + 3:10 * k + 6, i], terrain[10 * k + 6:10 * k + 9, i], terrain[10 * k:10 * k + 3, i]])


def contact_step_terrain(oracle, st, tau, push, terrain, plane_d, nsub, beta=0.2, eps=1e-8, margin=2e-3, obs_dt=0.0025):
    """One control period of every instance.  st: dict of SoA state arrays (base_pos, base_rot, base_rpy, base_vel, q, dq);
    tau [12, n], push [6, n], terrain [40, n], plane_d [4, n].  Returns (next state dict incl. foot_force, contact flags int [4, n],
    impulses of the last step [12, n] in the foot frames (t1, t2, n), 0 off contact)."""
    n = st["q"].shape[1]
    dt = obs_dt / nsub
    out = {k: np.array(st[k], dtype=np.float64) for k in STATE}
    out["foot_force"] = np.zeros((12, n))
    flags = np.zeros((4, n), dtype=np.int32)
    lam_out = np.zeros((12, n))
    for i in range(n):
        F = [frame(terrain, k, i) for k in range(4)]
        muk = terrain[9::10, i]
        cur = {k: out[k][:, i:i + 1].copy() for k in STATE}
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
            phi = np.array([F[k][:, 2] @ fp[k] for k in range(4)]) - plane_d[:, i]
            cand = [k for k in range(4) if phi[k] <= margin]
            lam = np.zeros(12)
            fl = np.zeros(4, dtype=np.int32)
            if cand:
                J = np.vstack([F[k].T @ Jall[3 * k:3 * k + 3] for k in cand])
                X = np.linalg.solve(M, J.T)
                G = J @ X
                H = G + eps * np.diag(np.diag(G))
                g = J @ nu
                for f, k in enumerate(cand):
                    g[3 * f + 2] += (1.0 if phi[k] >= 0.0 else beta) * phi[k] / dt
                A = np.zeros((5 * len(cand), 3 * len(cand)))
                for f, k in enumerate(cand):
                    A[5 * f:5 * f + 5, 3 * f:3 * f + 3] = pyramid_rows(muk[k])
                x, W, _ = primal_active_set(H, g, A)
                for f, k in enumerate(cand):
                    rows = {r - 5 * f for r in W if 5 * f <= r < 5 * f + 5}
                    lk = x[3 * f:3 * f + 3].copy()
                    if 0 in rows or (muk[k] > 0.0 and ({1, 2} <= rows or {3, 4} <= rows)) or lk[2] <= 0.0:
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
        for k in STATE:
            out[k][:, i] = cur[k][:, 0]
        for k in range(4):
            out["foot_force"][3 * k:3 * k + 3, i] = fR[k].T @ (F[k] @ lam[3 * k:3 * k + 3]) / dt
        flags[:, i] = fl
        lam_out[:, i] = lam
    return out, flags, lam_out
