"""Deterministic synthetic inputs for the batched WBC control cycle (SURVEY.md section 8d).

Stands in for the reference's Gazebo / ROS / TOWR layers (L5-L3): robot states, desired CoM and
swing-foot trajectory samples, contact modes, contact-sensor forces, pushes and terrain frames.
All arrays are SoA: shape [k, n] float64 (component-major), `mode` is int32 [n].

Randomness: numpy Philox, keyed by (seed, block) with blocks of 4096 instances, so instance i gets
the same numbers whatever the batch size or the number of ranks that shard the batch.

DoF order (canonical, tools/gen_model.py): [roll BL, BR, FL, FR, BL pitch, BL knee, BR pitch,
BR knee, FL pitch, FL knee, FR pitch, FR knee].  Stacked foot order: BR, BL, FL, FR (main.cpp:674-686).
"""
import numpy as np

BLOCK = 4096
MODE_STANCE, MODE_SWING_BR_FL, MODE_SWING_BL_FR = 0, 1, 2
TOTAL_MASS = 21.261

# nominal stand (main.cpp:1977-1988, 2001), canonical DoF order
Q_NOMINAL = np.array([0.000488, 0.000624, -3.2e-05, -0.000513,
                      -0.88425, -1.60390, 0.88620, 1.60326,
                      -0.88481, -1.60396, 0.88635, 1.60361])
BASE_Z_NOMINAL = 0.430159
# controller joint limits (main.cpp:612-613)
QMIN = np.array([-1.75, -1.75, -1.75, -1.75, -1.58, -2.62, -3.15, -0.02, -1.58, -2.62, -3.15, -0.02])
QMAX = np.array([1.75, 1.75, 1.75, 1.75, 3.15, 0.02, 1.58, 2.62, 3.15, 0.02, 1.58, 2.62])

# leg geometry (urdf:180-325 etc.), legs BL, BR, FL, FR
_HIP_XYZ = np.array([[-0.088, -0.2875, 0.0], [0.088, -0.2875, 0.0], [-0.088, 0.2875, 0.0], [0.088, 0.2875, 0.0]])
_ROLL_AXIS = np.array([[0, -1.0, 0], [0, -1.0, 0], [0, 1.0, 0], [0, 1.0, 0]])
_PITCH_XYZ = np.array([[-0.09875, 0, 0], [0.09875, 0, 0], [-0.09875, 0, 0], [0.09875, 0, 0]])
_PITCH_AXIS = np.array([[-1.0, 0, 0], [1.0, 0, 0], [-1.0, 0, 0], [1.0, 0, 0]])
_KNEE_XYZ = np.array([0.0, 0.0, -0.315])
_KNEE_AXIS = np.array([[1.0, 0, 0], [-1.0, 0, 0], [1.0, 0, 0], [-1.0, 0, 0]])
_FOOT_XYZ = np.array([-2.059009593607686e-05, -0.016585135985853, -0.321099633029770])
_LINK_M = np.array([0.836, 1.851, 0.302, 0.001])
_LINK_COM = [np.array([[-0.0074, 0, 0], [0.0074, 0, 0], [-0.0074, 0, 0], [0.0074, 0, 0]]),
             np.array([[-0.0418, 0, -0.0517], [0.0418, 0, -0.0517], [-0.0418, 0, -0.0517], [0.0418, 0, -0.0517]]),
             np.tile(np.array([0, -0.029, -0.1439]), (4, 1))]
_FOOT_LEG = [1, 0, 2, 3]   # stacked foot -> leg


def _rot_axis(axis, th):
    """Rodrigues rotation, axis [3], th [n] -> [n,3,3]."""
    a = np.asarray(axis, dtype=np.float64)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    s, c = np.sin(th)[:, None, None], np.cos(th)[:, None, None]
    return np.eye(3)[None] + s * K[None] + (1 - c) * (K @ K)[None]


def rpy_to_rot(rpy):
    """Fixed-axis XYZ (tf getRPY convention, main.cpp:436-446): R = Rz(yaw) Ry(pitch) Rx(roll). rpy [3,n] -> [n,3,3]."""
    r, p, y = rpy
    return _rot_axis([0, 0, 1], y) @ _rot_axis([0, 1, 0], p) @ _rot_axis([1, 0, 0], r)


def forward_kinematics(base_pos, base_rot, q):
    """Positions only (numpy, vectorised): returns (com [n,3], foot_pos [n,4,3] stacked BR,BL,FL,FR).

    base_pos [3,n], base_rot [9,n] row-major, q [12,n].  An independent restatement used to place
    desired trajectories near the actual CoM / feet and as a cross-check in the tests.
    """
    n = q.shape[1]
    R0 = base_rot.T.reshape(n, 3, 3)
    p0 = base_pos.T
    msum = np.full(n, 9.301)
    com = 9.301 * p0
    feet = np.zeros((n, 4, 3))
    for leg in range(4):
        R1 = R0 @ _rot_axis(_ROLL_AXIS[leg], q[leg])
        p1 = p0 + np.einsum("nij,j->ni", R0, _HIP_XYZ[leg])
        R2 = R1 @ _rot_axis(_PITCH_AXIS[leg], q[4 + 2 * leg])
        p2 = p1 + np.einsum("nij,j->ni", R1, _PITCH_XYZ[leg])
        R3 = R2 @ _rot_axis(_KNEE_AXIS[leg], q[5 + 2 * leg])
        p3 = p2 + np.einsum("nij,j->ni", R2, _KNEE_XYZ)
        pf = p3 + np.einsum("nij,j->ni", R3, _FOOT_XYZ)
        for m, R, p, c in ((_LINK_M[0], R1, p1, _LINK_COM[0][leg]), (_LINK_M[1], R2, p2, _LINK_COM[1][leg]),
                           (_LINK_M[2], R3, p3, _LINK_COM[2][leg]), (_LINK_M[3], R3, pf, np.zeros(3))):
            com = com + m * (p + np.einsum("nij,j->ni", R, c))
            msum = msum + m
        feet[:, _FOOT_LEG.index(leg), :] = pf
    return com / msum[:, None], feet


def _rng(seed, block, stream):
    return np.random.Generator(np.random.Philox(key=[int(seed) & 0xFFFFFFFFFFFFFFFF, (int(block) << 8) | int(stream)]))


def _block(seed, blk, cnt, mode_mix, pushes, terrain):
    g = lambda s: _rng(seed, blk, s)
    n = cnt
    sc = {}
    xy = g(0).uniform(-1.0, 1.0, (2, n))
    xy[xy == 0.0] = 0.25                                    # never the all-zero base position (main.cpp:584-588)
    z = g(1).uniform(0.36, 0.44, (1, n))
    sc["base_pos"] = np.vstack([xy, z])
    rpy = g(2).normal(0.0, 0.05, (3, n))
    sc["base_rpy"] = rpy
    R = rpy_to_rot(rpy)
    sc["base_rot"] = np.ascontiguousarray(R.reshape(n, 9).T)
    sc["base_vel"] = g(3).normal(0.0, 0.1, (6, n))
    q = Q_NOMINAL[:, None] + g(4).normal(0.0, 0.05, (12, n))
    sc["q"] = np.clip(q, QMIN[:, None], QMAX[:, None])
    sc["dq"] = g(5).normal(0.0, 0.5, (12, n))
    com, feet = forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T + g(6).normal(0.0, 0.02, (3, n)), rpy + g(7).normal(0.0, 0.02, (3, n))])
    sc["com_des_vel"] = g(8).normal(0.0, 0.05, (6, n))
    sc["com_des_acc"] = g(9).normal(0.0, 0.5, (6, n))
    u = g(10).uniform(0.0, 1.0, n)
    mode = np.full(n, MODE_STANCE, dtype=np.int32)
    mode[u >= mode_mix[0]] = MODE_SWING_BR_FL
    mode[u >= mode_mix[0] + mode_mix[1]] = MODE_SWING_BL_FR
    sc["mode"] = mode
    # contact-sensor forces (sensor frame), stacked BR,BL,FL,FR
    ff = np.zeros((12, n))
    fz = TOTAL_MASS * 9.81 / 4.0 * g(11).uniform(0.7, 1.3, (4, n))
    fxy = g(12).normal(0.0, 5.0, (8, n))
    for f in range(4):
        ff[3 * f + 0], ff[3 * f + 1], ff[3 * f + 2] = fxy[2 * f], fxy[2 * f + 1], fz[f]
    if pushes:
        # force_plugin case-4/5 law (fp.cpp:203-310): Fx = +-(5 + U{0..19}), Fy = +-(5 + U{0..9}) on one leg
        gp = g(13)
        leg = gp.integers(0, 4, n)
        fx = (5.0 + gp.integers(0, 20, n)) * gp.choice([-1.0, 1.0], n)
        fy = (5.0 + gp.integers(0, 10, n)) * gp.choice([-1.0, 1.0], n)
        idx = np.arange(n)
        ff[3 * leg + 0, idx] += fx
        ff[3 * leg + 1, idx] += fy
    sc["foot_force"] = ff
    # swing-foot references: the two swing feet in Jsw row order (mode 1: BR,FL = stacked 0,2; mode 2: BL,FR = 1,3)
    first = np.where(mode == MODE_SWING_BL_FR, 1, 0)
    second = np.where(mode == MODE_SWING_BL_FR, 3, 2)
    idx = np.arange(n)
    swp = np.hstack([feet[idx, first, :], feet[idx, second, :]]).T        # [6,n]
    arc = np.zeros((6, n))
    arc[2] = arc[5] = 0.06 * g(14).uniform(0.0, 1.0, n)                    # up to the 6 cm apex
    sc["sw_des_pos"] = swp + arc + g(15).normal(0.0, 0.01, (6, n))
    sc["sw_des_vel"] = g(16).normal(0.0, 0.2, (6, n))
    sc["sw_des_acc"] = g(17).normal(0.0, 2.0, (6, n))
    sc["obs_yd"] = g(18).normal(0.0, 0.5, (6, n))
    sc["obs_yw"] = g(19).normal(0.0, 0.1, (6, n))
    if terrain:
        gt = g(20)
        tr = np.zeros((40, n))
        for f in range(4):
            # unit normal uniform on the <=15 deg cap, tangents by Gram-Schmidt from x / y, mu in U(0.4, 0.8)
            cosmin = np.cos(np.deg2rad(15.0))
            ct = gt.uniform(cosmin, 1.0, n)
            st = np.sqrt(1.0 - ct * ct)
            ph = gt.uniform(0.0, 2 * np.pi, n)
            nrm = np.vstack([st * np.cos(ph), st * np.sin(ph), ct])
            t1 = np.array([1.0, 0, 0])[:, None] - nrm * nrm[0]
            t1 /= np.linalg.norm(t1, axis=0)
            t2 = np.cross(nrm.T, t1.T).T
            tr[10 * f + 0:10 * f + 3] = nrm
            tr[10 * f + 3:10 * f + 6] = t1
            tr[10 * f + 6:10 * f + 9] = t2
            tr[10 * f + 9] = gt.uniform(0.4, 0.8, n)
        sc["terrain"] = tr
    return sc


# BASELINE.json configs -> (mode mix stance/swingA/swingB, pushes, terrain, seed)
CONFIGS = {
    "standing_4096": dict(n=4096, mode_mix=(1.0, 0.0, 0.0), pushes=False, terrain=False, seed=1),
    "trot_65536": dict(n=65536, mode_mix=(0.25, 0.375, 0.375), pushes=True, terrain=False, seed=2),
    "mixed_terrain_1m": dict(n=1048576, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=True, seed=3),
}


def make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, terrain=False, seed=1, start=0):
    """Instances [start, start+n) of the infinite per-seed instance stream."""
    if n <= 0:
        sc = _block(seed, 0, 1, mode_mix, pushes, terrain)
        return {k: v[..., :0] for k, v in sc.items()}
    parts = []
    b0, b1 = start // BLOCK, (start + n - 1) // BLOCK
    for blk in range(b0, b1 + 1):
        sc = _block(seed, blk, BLOCK, mode_mix, pushes, terrain)
        lo = max(start, blk * BLOCK) - blk * BLOCK
        hi = min(start + n, (blk + 1) * BLOCK) - blk * BLOCK
        parts.append({k: v[..., lo:hi] for k, v in sc.items()})
    return {k: np.ascontiguousarray(np.concatenate([p[k] for p in parts], axis=-1)) for k in parts[0]}


def terrain_frames(normals, mu, feet=None):
    """Per-foot contact planes in the controller's terrain layout, so that one description feeds both the controller
    (`terrain` of a cycle) and the contact plant (WbcBatch.plant_contact_step(terrain=..., plane_d=...)).

    normals [4, 3, n] (or [3, n], the same for every foot; normalised here); mu a scalar, [n] or [4, n].  t1 is the world x axis
    projected onto the plane (the y axis where the normal is within 26 deg of x), t2 = n x t1.  feet [n, 4, 3]
    (forward_kinematics) puts each foot's plane through that foot point; None puts every plane through the origin.
    Returns (terrain [40, n], plane_d [4, n])."""
    nrm = np.asarray(normals, dtype=np.float64)
    if nrm.ndim == 2:
        nrm = np.broadcast_to(nrm, (4,) + nrm.shape)
    n = nrm.shape[2]
    mu = np.broadcast_to(np.asarray(mu, dtype=np.float64), (4, n))
    terrain, plane_d = np.zeros((40, n)), np.zeros((4, n))
    for f in range(4):
        nf = nrm[f] / np.linalg.norm(nrm[f], axis=0)
        near_x = np.abs(nf[0]) > 0.9
        axis = np.where(near_x, np.array([0.0, 1.0, 0.0])[:, None], np.array([1.0, 0.0, 0.0])[:, None])
        t1 = axis - nf * np.sum(axis * nf, axis=0)
        t1 /= np.linalg.norm(t1, axis=0)
        t2 = np.cross(nf.T, t1.T).T
        terrain[10 * f:10 * f + 3], terrain[10 * f + 3:10 * f + 6], terrain[10 * f + 6:10 * f + 9] = nf, t1, t2
        terrain[10 * f + 9] = mu[f]
        if feet is not None:
            plane_d[f] = np.sum(nf * feet[:, f, :].T, axis=0)
    return terrain, plane_d


def slope_terrain(feet, slope, azimuth, mu):
    """One slope per robot: the normal tilted by `slope` (rad) toward the downhill azimuth `azimuth` (rad from the world x axis),
    so that the ground falls by tan(slope) per metre along (cos azimuth, sin azimuth, 0), with friction mu (scalars or [n]).  Each
    foot's plane has that normal and passes through the foot's current point (feet [n, 4, 3]); four feet that do not lie on one
    such plane stand on parallel ones.  Returns (terrain [40, n], plane_d [4, n]), as terrain_frames."""
    n = feet.shape[0]
    sl, az = np.broadcast_to(np.asarray(slope, dtype=np.float64), (n,)), np.broadcast_to(np.asarray(azimuth, dtype=np.float64), (n,))
    nrm = np.vstack([np.sin(sl) * np.cos(az), np.sin(sl) * np.sin(az), np.cos(sl)])
    return terrain_frames(nrm, mu, feet)


SWEEP_DIRECTIONS, SWEEP_MAGNITUDES = 16, (5.0, 10.0, 20.0, 30.0, 40.0, 50.0, 65.0, 80.0)
SWEEP_GAINS = (1.0, 2.0, 5.0, 10.0, 20.0, 50.0, 100.0, 200.0)
SWEEP_STATES = 256


def push_sweep(n=None, start=0, directions=SWEEP_DIRECTIONS, magnitudes=SWEEP_MAGNITUDES, gains=SWEEP_GAINS, states=SWEEP_STATES, seed=4):
    """BASELINE config 5 (SURVEY.md 8d row 5): disturbance-rejection sweep.  The grid is
    directions x magnitudes x observer gains x states = 16 x 8 x 8 x 256 = 262144 standing instances; instance
    i = ((d * M + m) * G + g) * S + s.  The push is a horizontal force of the given magnitude (5..80 N, the range of
    force_plugin's case studies, fp.cpp:157, 206) in direction 2 pi d / D applied at the hip of leg (d mod 4), i.e. a
    world wrench [F; r x F] at the CoM.  Joints are at rest (dq = 0: the plant of this config is a CoM momentum
    integrator with locked joints), the observer starts from yd = yw = 0 and the measured foot forces carry the
    robot's weight.  Returns the scenario plus "obs_gain" [n], "push" [6,n] and "grid" (d, m, g, s index arrays).
    Instances [start, start+n) of the grid (default: all)."""
    D, M, G, S = int(directions), len(magnitudes), len(gains), int(states)
    total = D * M * G * S
    n = total - start if n is None else int(n)
    idx = start + np.arange(n)
    s_i = idx % S
    g_i = (idx // S) % G
    m_i = (idx // (S * G)) % M
    d_i = (idx // (S * G * M)) % D
    # the states: block-seeded like make(), indexed by s only, so that every grid cell sees the same 256 robots
    base = make(S, mode_mix=(1.0, 0.0, 0.0), pushes=False, terrain=False, seed=seed, start=0)
    sc = {k: np.ascontiguousarray(v[..., s_i]) for k, v in base.items()}
    sc["dq"] = np.zeros((12, n))
    sc["base_vel"] = np.zeros((6, n))
    sc["com_des_vel"] = np.zeros((6, n))
    sc["com_des_acc"] = np.zeros((6, n))
    sc["obs_yd"] = np.zeros((6, n))
    sc["obs_yw"] = np.zeros((6, n))
    # weight carried equally, expressed in the sensor (foot link) frame of a level robot: close enough to start from
    ff = np.zeros((12, n))
    ff[2::3] = TOTAL_MASS * 9.81 / 4.0
    sc["foot_force"] = ff
    com, _ = forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    ang = 2.0 * np.pi * d_i / D
    mag = np.asarray(magnitudes, dtype=np.float64)[m_i]
    F = np.vstack([mag * np.cos(ang), mag * np.sin(ang), np.zeros(n)])
    R0 = sc["base_rot"].T.reshape(n, 3, 3)
    hip = sc["base_pos"].T + np.einsum("nij,nj->ni", R0, _HIP_XYZ[d_i % 4])
    r = hip - com
    sc["push"] = np.vstack([F, np.cross(r, F.T).T])
    sc["obs_gain"] = np.asarray(gains, dtype=np.float64)[g_i]
    sc["grid"] = np.vstack([d_i, m_i, g_i, s_i])
    return sc


def make_config(name, n=None, start=0):
    cfg = dict(CONFIGS[name])
    n_cfg = cfg.pop("n")
    return make(n if n is not None else n_cfg, start=start, **cfg)


def trot_replay(cycles_per_phase=46, seed=0x0D06B07):
    """Config 1: ONE DogBot replaying 4 gait phases (stance, swing{BR,FL}, stance, swing{BL,FR}) of a
    synthetic trot (SURVEY.md 8d row 1).  Returns a scenario whose instance index is the cycle index;
    observer state must be chained by the caller (cycle k+1 uses the state produced by cycle k)."""
    n = 4 * cycles_per_phase
    t = np.arange(n) * 0.0025
    sc = {}
    sway = 0.02 * np.sin(2 * np.pi * 1.0 * t)
    sc["base_pos"] = np.vstack([0.3 + sway, -0.2 + 0.5 * sway, np.full(n, BASE_Z_NOMINAL)])
    rpy = np.vstack([0.01 * np.sin(2 * np.pi * 1.5 * t), 0.01 * np.cos(2 * np.pi * 1.2 * t), 0.05 * np.ones(n)])
    sc["base_rpy"] = rpy
    sc["base_rot"] = np.ascontiguousarray(rpy_to_rot(rpy).reshape(n, 9).T)
    dsway = 0.02 * 2 * np.pi * np.cos(2 * np.pi * t)
    sc["base_vel"] = np.vstack([dsway, 0.5 * dsway, np.zeros(n), 0.01 * 2 * np.pi * 1.5 * np.cos(2 * np.pi * 1.5 * t),
                                -0.01 * 2 * np.pi * 1.2 * np.sin(2 * np.pi * 1.2 * t), np.zeros(n)])
    ph = np.linspace(0, 2 * np.pi, 12, endpoint=False)[:, None]
    sc["q"] = np.clip(Q_NOMINAL[:, None] + 0.1 * np.sin(2 * np.pi * 2.0 * t[None, :] + ph), QMIN[:, None], QMAX[:, None])
    sc["dq"] = 0.1 * 2 * np.pi * 2.0 * np.cos(2 * np.pi * 2.0 * t[None, :] + ph)
    com, feet = forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    # desired CoM: cubic Hermite from the initial CoM to +4 cm in x over 0.5 s (mimics main.cpp:925-940)
    s = np.clip(t / 0.5, 0, 1)
    hp, hv, ha = 3 * s ** 2 - 2 * s ** 3, (6 * s - 6 * s ** 2) / 0.5, (6 - 12 * s) / 0.25
    p0 = np.array([com[0, 0], com[0, 1], 0.4])
    des = np.zeros((6, n)); dv = np.zeros((6, n)); da = np.zeros((6, n))
    des[0:3] = p0[:, None]; des[0] += 0.04 * hp; dv[0] = 0.04 * hv; da[0] = 0.04 * ha
    des[5] = rpy[2]
    sc["com_des_pos"], sc["com_des_vel"], sc["com_des_acc"] = des, dv, da
    mode = np.repeat(np.array([MODE_STANCE, MODE_SWING_BR_FL, MODE_STANCE, MODE_SWING_BL_FR], dtype=np.int32),
                     cycles_per_phase)
    sc["mode"] = mode
    rng = _rng(seed, 0, 0)
    ff = np.zeros((12, n))
    for f in range(4):
        ff[3 * f + 2] = TOTAL_MASS * 9.81 / 4.0 * (1.0 + 0.1 * np.sin(2 * np.pi * 3 * t + f))
        ff[3 * f + 0] = 2.0 * np.sin(2 * np.pi * 2 * t + f)
        ff[3 * f + 1] = 2.0 * np.cos(2 * np.pi * 2 * t + f)
    sc["foot_force"] = ff + rng.normal(0, 0.1, (12, n))
    first = np.where(mode == MODE_SWING_BL_FR, 1, 0)
    second = np.where(mode == MODE_SWING_BL_FR, 3, 2)
    idx = np.arange(n)
    swp = np.hstack([feet[idx, first, :], feet[idx, second, :]]).T
    phase_t = (np.arange(n) % cycles_per_phase) / cycles_per_phase
    arc = np.zeros((6, n)); arc[2] = arc[5] = 0.06 * np.sin(np.pi * phase_t) ** 2
    sc["sw_des_pos"] = swp + arc
    sc["sw_des_vel"] = np.zeros((6, n)); sc["sw_des_acc"] = np.zeros((6, n))
    sc["obs_yd"] = np.zeros((6, n)); sc["obs_yw"] = np.zeros((6, n))
    return sc


def make_trajectory(sc, nseg=3, seed=11, match_acc=False):
    """A synthetic plan for the n instances of scenario `sc` in the table layout of wbc_set_trajectory (SURVEY.md 8f-1):
    four splines (base_linear, base_angular, two swing feet) of `nseg` cubic-Hermite polynomials each, starting at the
    scenario's desired CoM pose / swing-foot targets, plus sample times t [n] inside the plan.  Every 5th instance is
    sampled exactly on a junction of spline 0 (towr returns the previous polynomial there, spline.cc:48-66), every 7th
    at t = 0.  match_acc: choose the second node of every spline so that the acceleration at t = 0 equals the scenario's
    desired acceleration too (p1 = p0 + (a0 T^2 / 2 + 2 T v0) / 3, v1 = 0): sampled at t = 0 the plan then reproduces
    the scenario's 36 desired-trajectory inputs (positions and velocities bit for bit, accelerations to rounding)."""
    n = int(sc["mode"].shape[0])
    rng = np.random.Generator(np.random.Philox(key=[seed, 0x7261]))
    dur = rng.uniform(0.1, 0.5, size=(4 * nseg, n))
    nodes = np.zeros((4 * (nseg + 1) * 6, n))
    accs = [sc["com_des_acc"][0:3], sc["com_des_acc"][3:6], sc["sw_des_acc"][0:3], sc["sw_des_acc"][3:6]]
    starts = [(sc["com_des_pos"][0:3], sc["com_des_vel"][0:3], 0.02, 0.05), (sc["com_des_pos"][3:6], sc["com_des_vel"][3:6], 0.03, 0.1),
              (sc["sw_des_pos"][0:3], sc["sw_des_vel"][0:3], 0.03, 0.3), (sc["sw_des_pos"][3:6], sc["sw_des_vel"][3:6], 0.03, 0.3)]
    for s, (p0, v0, sp, sv) in enumerate(starts):
        p, v = np.array(p0, dtype=np.float64), np.array(v0, dtype=np.float64)
        for k in range(nseg + 1):
            r = (s * (nseg + 1) + k) * 6
            nodes[r:r + 3], nodes[r + 3:r + 6] = p, v
            if match_acc and k == 0:
                T = dur[s * nseg]
                p = p + (accs[s] * T * T / 2.0 + 2.0 * T * v) / 3.0
                v = np.zeros((3, n))
                continue
            p = p + rng.normal(0.0, sp, size=(3, n))
            v = rng.normal(0.0, sv, size=(3, n))
    total = np.min([dur[s * nseg:(s + 1) * nseg].sum(axis=0) for s in range(4)], axis=0)
    t = rng.uniform(0.0, 1.0, size=n) * total
    idx = np.arange(n)
    j = idx % nseg
    junction = np.cumsum(dur[0:nseg], axis=0)[j, idx]
    on_j = (idx % 5 == 0) & (junction <= total)
    t[on_j] = junction[on_j]
    t[idx % 7 == 0] = 0.0
    return {"nseg": nseg, "durations": np.ascontiguousarray(dur), "nodes": np.ascontiguousarray(nodes), "t": t}


ROLLOUT_CYCLES_PER_PHASE = 46      # 0.115 s per gait phase at the 400 Hz control rate (quadruped_gait_generator.cc:277-310 durations, main.cpp:861)


def _rollout_constants(n, start, seed):
    """Per-robot constants of trot_rollout, block-keyed like make(): robot i gets the same numbers whatever the batch size
    or the number of ranks."""
    parts = []
    b0, b1 = start // BLOCK, (start + max(n, 1) - 1) // BLOCK
    for blk in range(b0, b1 + 1):
        g = lambda s: _rng(seed, blk, s)
        c = {"phase": g(0).integers(0, 4 * ROLLOUT_CYCLES_PER_PHASE, BLOCK),
             "xy": g(1).uniform(-1.0, 1.0, (2, BLOCK)), "yaw": g(2).uniform(-0.3, 0.3, BLOCK),
             "amp": g(3).uniform(0.04, 0.12, (12, BLOCK)), "freq": g(4).uniform(1.5, 2.5, BLOCK),
             "ph": g(5).uniform(0.0, 2 * np.pi, (12, BLOCK)), "sway": g(6).uniform(0.005, 0.03, BLOCK),
             "z": g(7).uniform(0.40, 0.44, BLOCK), "des": g(8).uniform(0.0, 2 * np.pi, (6, BLOCK)),
             "push_leg": g(9).integers(0, 4, BLOCK), "push_fx": (5.0 + g(10).integers(0, 20, BLOCK)) * g(11).choice([-1.0, 1.0], BLOCK),
             "push_fy": (5.0 + g(12).integers(0, 10, BLOCK)) * g(13).choice([-1.0, 1.0], BLOCK),
             "push_t0": g(14).integers(0, 4 * ROLLOUT_CYCLES_PER_PHASE, BLOCK)}
        c["xy"][c["xy"] == 0.0] = 0.25
        lo = max(start, blk * BLOCK) - blk * BLOCK
        hi = min(start + n, (blk + 1) * BLOCK) - blk * BLOCK
        parts.append({k: v[..., lo:hi] for k, v in c.items()})
    return {k: np.concatenate([p[k] for p in parts], axis=-1) for k in parts[0]}


def trot_rollout(n, step, seed=5, start=0):
    """Evolving-state workload: robots [start, start+n) of a herd that trots through the gait cycle of configs[0]
    (stance, swing{BR,FL}, stance, swing{BL,FR}; 46 control cycles each, main.cpp:978-1400 phase switching) with
    per-robot phase offsets, gaits and pushes.  Returns the inputs of control cycle `step` (0, 1, 2, ...) for every robot:
    robot r is at cycle k = phase_r + step of its own gait, so at any step a quarter of the herd changes contact mode
    within the next 11 cycles, swing and stance solves are mixed, and the QP active sets drift from cycle to cycle.
    The observer state is NOT part of the scenario: the caller chains it (cycle k+1 uses the state cycle k produced).
    A force_plugin-style push (fp.cpp:203-310: Fx = +-(5..24) N, Fy = +-(5..14) N on one leg) acts on each robot for 40
    cycles of every gait cycle and shows up in the measured force of that leg."""
    C = _rollout_constants(n, start, seed)
    cpp = ROLLOUT_CYCLES_PER_PHASE
    k = C["phase"] + int(step)
    t = k * 0.0025
    w = 2 * np.pi * C["freq"]
    sc = {}
    sway = C["sway"] * np.sin(2 * np.pi * 1.0 * t)
    dsway = C["sway"] * 2 * np.pi * np.cos(2 * np.pi * 1.0 * t)
    sc["base_pos"] = np.vstack([C["xy"][0] + sway, C["xy"][1] + 0.5 * sway, C["z"]])
    rpy = np.vstack([0.01 * np.sin(2 * np.pi * 1.5 * t), 0.01 * np.cos(2 * np.pi * 1.2 * t), C["yaw"]])
    sc["base_rpy"] = rpy
    sc["base_rot"] = np.ascontiguousarray(rpy_to_rot(rpy).reshape(n, 9).T)
    # world-frame base twist consistent with the scripted pose (yaw constant: the roll/pitch rates are the body rates to first order)
    sc["base_vel"] = np.vstack([dsway, 0.5 * dsway, np.zeros(n), 0.01 * 2 * np.pi * 1.5 * np.cos(2 * np.pi * 1.5 * t),
                                -0.01 * 2 * np.pi * 1.2 * np.sin(2 * np.pi * 1.2 * t), np.zeros(n)])
    arg = w[None, :] * t[None, :] + C["ph"]
    sc["q"] = np.clip(Q_NOMINAL[:, None] + C["amp"] * np.sin(arg), QMIN[:, None], QMAX[:, None])
    sc["dq"] = C["amp"] * w[None, :] * np.cos(arg)
    com, feet = forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    off = 0.015 * np.sin(2 * np.pi * 0.8 * t[None, :] + C["des"])
    sc["com_des_pos"] = np.vstack([com.T + off[0:3], rpy + 0.5 * off[3:6]])
    sc["com_des_vel"] = 0.015 * 2 * np.pi * 0.8 * np.cos(2 * np.pi * 0.8 * t[None, :] + C["des"]) * np.array([1, 1, 1, .5, .5, .5])[:, None]
    sc["com_des_acc"] = -0.015 * (2 * np.pi * 0.8) ** 2 * np.sin(2 * np.pi * 0.8 * t[None, :] + C["des"]) * np.array([1, 1, 1, .5, .5, .5])[:, None]
    phase = (k // cpp) % 4
    mode = np.array([MODE_STANCE, MODE_SWING_BR_FL, MODE_STANCE, MODE_SWING_BL_FR], dtype=np.int32)[phase]
    sc["mode"] = np.ascontiguousarray(mode)
    # measured foot forces (sensor frame, stacked BR,BL,FL,FR): the stance feet share the weight
    swing = np.zeros((4, n), dtype=bool)
    swing[0] = swing[2] = mode == MODE_SWING_BR_FL
    swing[1] = swing[3] = mode == MODE_SWING_BL_FR
    nst = 4 - swing.sum(axis=0)
    ff = np.zeros((12, n))
    for f in range(4):
        ff[3 * f + 2] = np.where(swing[f], 0.0, TOTAL_MASS * 9.81 / nst * (1.0 + 0.1 * np.sin(2 * np.pi * 3 * t + f)))
        ff[3 * f + 0] = np.where(swing[f], 0.0, 2.0 * np.sin(2 * np.pi * 2 * t + f))
        ff[3 * f + 1] = np.where(swing[f], 0.0, 2.0 * np.cos(2 * np.pi * 2 * t + f))
    pushing = ((k - C["push_t0"]) % (4 * cpp)) < 40
    idx = np.arange(n)
    ff[3 * C["push_leg"] + 0, idx] += np.where(pushing, C["push_fx"], 0.0)
    ff[3 * C["push_leg"] + 1, idx] += np.where(pushing, C["push_fy"], 0.0)
    sc["foot_force"] = ff
    first = np.where(mode == MODE_SWING_BL_FR, 1, 0)
    second = np.where(mode == MODE_SWING_BL_FR, 3, 2)
    swp = np.hstack([feet[idx, first, :], feet[idx, second, :]]).T
    phase_t = (k % cpp) / cpp
    arc = np.zeros((6, n)); arc[2] = arc[5] = 0.06 * np.sin(np.pi * phase_t) ** 2
    sc["sw_des_pos"] = swp + arc
    sc["sw_des_vel"] = np.zeros((6, n)); sc["sw_des_acc"] = np.zeros((6, n))
    return sc
