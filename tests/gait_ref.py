"""Independent numpy restatement of the trot gait law (DESIGN.md 4.8), written from the law's text rather than from
csrc/wbc_gait.cuh: feet and CoM from scenarios.forward_kinematics, hips from the URDF's hip-joint origins.  Vectorised over robots;
arrays are SoA [k, n] like the C ABI's.  Its choices, restated from the law:
  * the (vx, vy) ramp clips the 2-vector change to length acc_lin dt; the yaw-rate ramp clips to +-acc_yaw dt;
  * com_des_acc is the clipped change over dt, rotated into the world, plus omega z x v_w; row 5 the yaw-rate change over dt;
  * the emitted yaw is yaw_meas + wrap(yaw_ref - yaw_meas), wrap(a) = a - 2 pi floor((a + pi) / (2 pi));
  * in a swing phase the swing curve is emitted even after touchdown; in a stance phase the current points of the pair that swings
    next, with zero velocity and acceleration;
  * ground height under (x, y) = mean of the four feet's plane heights (d_k - n_x x - n_y y) / n_z; 0 on flat ground;
  * init: k0 modulo the gait period; robots in a stance phase get liftoff = target = the current points of the next swing pair."""
import numpy as np

from wbc_quadruped_dob_b200 import scenarios as S

HIP = np.array([[-0.088, -0.2875, 0.0], [0.088, -0.2875, 0.0], [-0.088, 0.2875, 0.0], [0.088, 0.2875, 0.0]])   # legs BL, BR, FL, FR
FOOT_LEG = (1, 0, 2, 3)                 # stacked BR, BL, FL, FR -> leg
TOUCHDOWN_S = 0.5
ST_BAD_MODE, ST_NONFINITE, ST_BAD_TERRAIN = -20, -21, -24
OUT = ("com_des_pos", "com_des_vel", "com_des_acc", "sw_des_pos", "sw_des_vel", "sw_des_acc")


def kinematics(st):
    """(com [n, 3], hips [n, 4, 3], feet [n, 4, 3]) in stacked foot order."""
    com, feet = S.forward_kinematics(st["base_pos"], st["base_rot"], st["q"])
    n = com.shape[0]
    R = st["base_rot"].T.reshape(n, 3, 3)
    hips = np.stack([st["base_pos"].T + R @ HIP[FOOT_LEG[f]] for f in range(4)], axis=1)
    return com, hips, feet


def _planes(terrain, plane_d, n):
    if terrain is None:
        return None
    nrm = np.stack([terrain[10 * f:10 * f + 3] for f in range(4)])          # [4, 3, n]
    d = np.zeros((4, n)) if plane_d is None else plane_d
    return nrm, d


def _plane_z(pl, f, x, y):
    nrm, d = pl
    return (d[f] - nrm[f, 0] * x - nrm[f, 1] * y) / nrm[f, 2]


def _ground(pl, x, y):
    if pl is None:
        return np.zeros_like(x)
    return 0.25 * (_plane_z(pl, 0, x, y) + _plane_z(pl, 1, x, y) + _plane_z(pl, 2, x, y) + _plane_z(pl, 3, x, y))


def _validate(st, terrain, plane_d, extra=()):
    n = st["q"].shape[1]
    arrs = [st["base_pos"], st["base_rot"], st["base_rpy"][2:3], st["base_vel"][0:3], st["q"]] + list(extra)
    ok = np.ones(n, bool)
    for a in arrs:
        ok &= np.isfinite(a).all(axis=0)
    frames = np.ones(n, bool)
    if terrain is not None:
        for f in range(4):
            F = terrain[10 * f:10 * f + 9].reshape(3, 3, n)           # rows n, t1, t2
            ok &= np.isfinite(F).all(axis=(0, 1))
            G = np.einsum("ain,bin->abn", F, F)
            frames &= (np.abs(G - np.eye(3)[:, :, None]) <= 1e-9).all(axis=(0, 1)) & (F[0, 2] >= 0.5)
        if plane_d is not None:
            ok &= np.isfinite(plane_d).all(axis=0)
    return np.where(~ok, ST_NONFINITE, np.where(~frames, ST_BAD_TERRAIN, 0)).astype(np.int32)


def _pair(phase):
    return np.where(phase < 2, 0, 1), np.where(phase < 2, 2, 3)


def _target(G, dt, f, hip, p0z, cref, vref, off, vmeas, pl):
    """Touchdown targets [n, 3] of stacked feet f [n] (hip [n, 3])."""
    n = hip.shape[0]
    idx = np.arange(n)
    tau = G["swing_cycles"] * dt + (2 * G["stance_cycles"] + G["swing_cycles"]) * dt / 2.0
    cy, sy = np.cos(cref[3]), np.sin(cref[3])
    vw = np.stack([cy * vref[0] - sy * vref[1], sy * vref[0] + cy * vref[1]])
    r = hip[:, :2].T - cref[0:2]
    turn = np.stack([-vref[2] * r[1], vref[2] * r[0]])
    o = off[2 * f, idx], off[2 * f + 1, idx]
    neutral = hip[:, :2].T + tau * (vw + turn) + np.stack([cy * o[0] - sy * o[1], sy * o[0] + cy * o[1]])
    corr = G["k_v"] * (vmeas[0:2] - vw)
    nc = np.sqrt(corr[0] ** 2 + corr[1] ** 2)
    scale = np.where(nc > G["max_step"], G["max_step"] / np.where(nc > 0, nc, 1.0), 1.0)
    xy = neutral + corr * scale
    z = p0z.copy()
    if pl is not None:
        nrm, d = pl
        z = (d[f, idx] - nrm[f, 0, idx] * xy[0] - nrm[f, 1, idx] * xy[1]) / nrm[f, 2, idx]
    return np.vstack([xy, z]).T


def init(G, dt, st, k0=None, terrain=None, plane_d=None):
    """Returns (gait state dict, status [n]); refused robots get zeros (the caller compares only accepted ones)."""
    n = st["q"].shape[1]
    status = _validate(st, terrain, plane_d)
    pl = _planes(terrain, plane_d, n)
    com, hips, feet = kinematics(st)
    yaw = st["base_rpy"][2]
    gs = {"com_ref": np.vstack([com[:, 0], com[:, 1], com[:, 2] - _ground(pl, com[:, 0], com[:, 1]), yaw]), "v_ref": np.zeros((3, n))}
    cy, sy = np.cos(yaw), np.sin(yaw)
    off = np.zeros((8, n))
    for f in range(4):
        d = feet[:, f, :2] - hips[:, f, :2]
        off[2 * f], off[2 * f + 1] = cy * d[:, 0] + sy * d[:, 1], -sy * d[:, 0] + cy * d[:, 1]
    gs["offset"] = off
    Ns, Nw = G["stance_cycles"], G["swing_cycles"]
    k = np.mod(np.zeros(n, np.int64) if k0 is None else np.asarray(k0, np.int64), 2 * (Ns + Nw))
    bounds = np.array([Ns, Ns + Nw, 2 * Ns + Nw])
    phase = np.searchsorted(bounds, k, side="right")
    start = np.concatenate([[0], bounds])[phase]
    gs["phase"], gs["tick"], gs["landed"] = phase[None].astype(np.int32), (k - start)[None].astype(np.int32), np.zeros((1, n), np.int32)
    idx = np.arange(n)
    lo, tg = np.zeros((6, n)), np.zeros((6, n))
    for j, f in enumerate(_pair(phase)):
        p0 = feet[idx, f, :]
        p1 = _target(G, dt, f, hips[idx, f, :], p0[:, 2], gs["com_ref"], gs["v_ref"], off, st["base_vel"], pl)
        p1 = np.where((phase % 2 == 1)[:, None], p1, p0)
        lo[3 * j:3 * j + 3], tg[3 * j:3 * j + 3] = p0.T, p1.T
    gs["liftoff"], gs["target"] = lo, tg
    for key in gs:
        gs[key][..., status != 0] = 0
    return gs, status


def step(G, dt, gs, st, cmd=None, contact=None, terrain=None, plane_d=None):
    """One gait step.  Returns (new gait state, outputs dict with "mode" and the six desired arrays, status [n]); refused robots keep
    their state and get zero outputs."""
    n = st["q"].shape[1]
    Ns, Nw = G["stance_cycles"], G["swing_cycles"]
    cmd = np.zeros((3, n)) if cmd is None else cmd
    gst = [gs[k] for k in ("com_ref", "v_ref", "liftoff", "target", "offset")]
    status = _validate(st, terrain, plane_d, extra=gst + [cmd])
    phase, tick, landed = gs["phase"][0].astype(np.int64), gs["tick"][0].astype(np.int64), gs["landed"][0].copy()
    swing = phase % 2 == 1
    length = np.where(swing, Nw, Ns)
    bad = (phase < 0) | (phase > 3) | (tick < 0) | (tick >= length)
    status = np.where((status == 0) & bad, ST_BAD_MODE, status).astype(np.int32)
    pl = _planes(terrain, plane_d, n)
    com, hips, feet = kinematics(st)
    idx = np.arange(n)
    f0, f1 = _pair(phase)
    # 1. touchdown
    if contact is not None:
        past = (tick + 1) / Nw > TOUCHDOWN_S
        landed = np.where(swing & (landed == 0) & past & (contact[f0, idx] != 0) & (contact[f1, idx] != 0), 1, landed)
    cref, vref = gs["com_ref"].copy(), gs["v_ref"].copy()
    p0, p1 = gs["liftoff"].copy(), gs["target"].copy()
    # 2. lift-off
    lift = swing & (tick == 0)
    for j, f in enumerate((f0, f1)):
        a = feet[idx, f, :]
        b = _target(G, dt, f, hips[idx, f, :], a[:, 2], cref, vref, gs["offset"], st["base_vel"], pl)
        p0[3 * j:3 * j + 3] = np.where(lift, a.T, p0[3 * j:3 * j + 3])
        p1[3 * j:3 * j + 3] = np.where(lift, b.T, p1[3 * j:3 * j + 3])
    # 3. command ramp
    dv = cmd[0:2] - vref[0:2]
    lim = G["acc_lin"] * dt
    dn = np.sqrt(dv[0] ** 2 + dv[1] ** 2)
    clip = dn > lim
    dv = np.where(clip, dv * (lim / np.where(clip, dn, 1.0)), dv)
    vref[0:2] = np.where(clip, vref[0:2] + dv, cmd[0:2])
    wlim = G["acc_yaw"] * dt
    dw = cmd[2] - vref[2]
    wclip = np.abs(dw) > wlim
    dw = np.clip(dw, -wlim, wlim)
    vref[2] = np.where(wclip, vref[2] + dw, cmd[2])
    # 4. CoM reference
    w = vref[2]
    cref[3] = cref[3] + w * dt
    cy, sy = np.cos(cref[3]), np.sin(cref[3])
    vw = np.stack([cy * vref[0] - sy * vref[1], sy * vref[0] + cy * vref[1]])
    cref[0:2] = cref[0:2] + vw * dt
    e = cref[0:2] - com[:, 0:2].T
    en = np.sqrt(e[0] ** 2 + e[1] ** 2)
    far = en > G["leash"]
    cref[0:2] = np.where(far, com[:, 0:2].T + e * (G["leash"] / np.where(far, en, 1.0)), cref[0:2])
    zref = cref[2] + _ground(pl, cref[0], cref[1])
    # 5. emit
    mode = np.where(landed != 0, S.MODE_STANCE, np.where(phase == 1, S.MODE_SWING_BR_FL, np.where(phase == 3, S.MODE_SWING_BL_FR, S.MODE_STANCE)))
    dyaw = cref[3] - st["base_rpy"][2]
    dyaw = dyaw - 2.0 * np.pi * np.floor((dyaw + np.pi) / (2.0 * np.pi))
    a = dv / dt
    z = np.zeros(n)
    out = {"mode": mode.astype(np.int32),
           "com_des_pos": np.vstack([cref[0], cref[1], zref, z, z, st["base_rpy"][2] + dyaw]),
           "com_des_vel": np.vstack([vw[0], vw[1], z, z, z, w]),
           "com_des_acc": np.vstack([cy * a[0] - sy * a[1] - w * vw[1], sy * a[0] + cy * a[1] + w * vw[0], z, z, z, dw / dt])}
    s = (tick + 1) / Nw
    r = 1.0 / (Nw * dt)
    sig, dsig, ddsig = 10 * s ** 3 - 15 * s ** 4 + 6 * s ** 5, (30 * s ** 2 - 60 * s ** 3 + 30 * s ** 4) * r, (60 * s - 180 * s ** 2 + 120 * s ** 3) * r * r
    up = np.zeros((6, 1)); up[2] = up[5] = G["step_height"]
    sp = p0 + (p1 - p0) * sig + up * np.sin(np.pi * s) ** 2
    sv = (p1 - p0) * dsig + up * np.pi * np.sin(2 * np.pi * s) * r
    sa = (p1 - p0) * ddsig + up * 2 * np.pi ** 2 * np.cos(2 * np.pi * s) * r * r
    stand = np.vstack([feet[idx, f0, :].T, feet[idx, f1, :].T])
    out["sw_des_pos"] = np.where(swing, sp, stand)
    out["sw_des_vel"] = np.where(swing, sv, 0.0)
    out["sw_des_acc"] = np.where(swing, sa, 0.0)
    # 6. advance
    tick = tick + 1
    end = tick >= length
    new = {"phase": np.where(end, (phase + 1) % 4, phase)[None].astype(np.int32), "tick": np.where(end, 0, tick)[None].astype(np.int32),
           "landed": np.where(end, 0, landed)[None].astype(np.int32), "com_ref": cref, "v_ref": vref, "liftoff": p0, "target": p1,
           "offset": gs["offset"].copy()}
    keep = status != 0
    for k in new:
        new[k][..., keep] = gs[k][..., keep]
    for k in out:
        out[k][..., keep] = 0
    return new, out, status
