"""The contact plant on inclined ground (wbc_plant_contact_step_terrain, the terrain form of csrc/wbc_contact.cuh): per-foot planes
n . p = d and friction from the controller's terrain frames.

CPU: the kernel's terrain instantiation compiled for the host (tests/host_emu/contact_terrain_emu.cpp) against the flat plant,
against itself in a rotated world, against the independent reference (tests/contact_ref_terrain.py), and closed through
the controller's host emulation on a slope and in a V-groove; refusals of bad frames.  GPU: the kernel against the emulation and
against the flat entry point, and a closed-loop trot of 4096 robots on their own slopes."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import contact_ref as CR
from tests import contact_ref_terrain as CRT
from tests import util
from tests.test_contact_plant import STATE, ContactEmu, _ContactParams, _standing, mixed_states
from wbc_quadruped_dob_b200 import scenarios as S

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
ST_NONFINITE, ST_BAD_TERRAIN = -21, -24


class TerrainEmu:
    """g++ build of contact_step_instance<true> (test infrastructure only)."""

    def __init__(self):
        so = os.path.join(util.EMU_DIR, "libcontact_terrain_emu.so")
        util._build_emu(os.path.join(util.EMU_DIR, "contact_terrain_emu.cpp"), so)
        self.lib = C.CDLL(so)
        self.lib.emu_contact_terrain_step.argtypes = [C.POINTER(util.EmuParams), C.POINTER(_ContactParams), C.c_int, C.c_long] + \
            [_dp] * 7 + [_dp, _dp, _dp, _dp, _ip, _dp, _ip, C.c_int]
        self.lib.emu_contact_terrain_step.restype = None

    def step(self, st, tau, push, terrain, plane_d=None, nsub=5, params=None, cp=(0.2, 1e-8, 2e-3, 64)):
        """Advances a copy of st; returns (next state incl. foot_force, contact [4, n], diag [4, n], status [n])."""
        n = st["q"].shape[1]
        P = params or util.emu_default_params()
        out = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
        out["foot_force"] = np.array(st.get("foot_force", np.zeros((12, n))), dtype=np.float64, order="C")
        contact, diag, status = np.zeros((4, n), np.int32), np.zeros((4, n)), np.zeros(n, np.int32)
        keep = [np.ascontiguousarray(a, dtype=np.float64) if a is not None else None for a in (tau, push, terrain, plane_d)]
        d = lambda a: None if a is None else a.ctypes.data_as(_dp)
        self.lib.emu_contact_terrain_step(C.byref(P), C.byref(_ContactParams(*cp)), n, n, *[d(out[k]) for k in STATE], d(out["foot_force"]),
                                          *[d(a) for a in keep], contact.ctypes.data_as(_ip), d(diag), status.ctypes.data_as(_ip), int(nsub))
        return out, contact, diag, status


@pytest.fixture(scope="module")
def cemu():
    return ContactEmu()


@pytest.fixture(scope="module")
def temu():
    return TerrainEmu()


def horizontal_terrain(mu, n):
    """n = e3, t1 = e1, t2 = e2 on every foot, mu [n] on all four feet."""
    tr = np.zeros((40, n))
    for f in range(4):
        tr[10 * f + 2] = tr[10 * f + 3] = tr[10 * f + 7] = 1.0
        tr[10 * f + 9] = mu
    return tr


def _rel(a, b):
    return np.abs(a - b).max() / max(1.0, np.abs(b).max())


def test_scenario_helpers_build_the_controllers_layout():
    """slope_terrain / terrain_frames: orthonormal right-handed frames, the downhill direction falls, planes through the feet."""
    sc = S.make(5, seed=3)
    _, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    tr, d = S.slope_terrain(feet, np.deg2rad(15.0), np.linspace(0.0, 6.0, 5), 0.6)
    for f in range(4):
        F = np.stack([tr[10 * f + 3:10 * f + 6], tr[10 * f + 6:10 * f + 9], tr[10 * f:10 * f + 3]])   # [3 (t1 t2 n), 3, n]
        for i in range(5):
            assert np.abs(F[:, :, i] @ F[:, :, i].T - np.eye(3)).max() < 1e-15
            assert abs(np.linalg.det(F[:, :, i]) - 1.0) < 1e-15
            assert abs(F[2, :, i] @ feet[i, f] - d[f, i]) < 1e-15
        assert np.allclose(np.arccos(F[2, 2]), np.deg2rad(15.0))
        assert (tr[10 * f + 9] == 0.6).all()
    az = np.linspace(0.0, 6.0, 5)
    assert np.allclose(tr[0] * np.cos(az) + tr[1] * np.sin(az), np.sin(np.deg2rad(15.0)))     # n leans downhill
    wall, _ = S.terrain_frames(np.array([[1.0], [0.0], [0.0]]), 0.5)                        # a normal along x takes t1 from y
    assert np.allclose(wall[3:6, 0], [0.0, 1.0, 0.0]) and np.allclose(wall[6:9, 0], [0.0, 0.0, 1.0])


def test_terrain_replaces_ground_z_and_mu():
    """plant_contact_step(terrain=...) refuses ground_z, mu, and plane_d without terrain, before it touches the library."""
    from wbc_quadruped_dob_b200 import api
    z4, z40 = np.zeros((4, 1)), np.zeros((40, 1))
    for kw in (dict(terrain=z40, ground_z=z4), dict(terrain=z40, mu=np.zeros(1)), dict(plane_d=z4)):
        with pytest.raises(ValueError):
            api.WbcBatch.plant_contact_step(None, {}, None, None, **kw)


# ------------------------------------------------------------------------------------------------------------ CPU: emulation
def test_horizontal_terrain_reproduces_the_flat_plant(cemu, temu):
    """n = e3, t1 = e1, t2 = e2, d = ground_z and each foot's mu the instance's: status and flags equal, state, foot_force and diag
    within 1e-14 (relative) of the flat plant on 512 mixed states with 1 and 5 substeps.  The rotation multiplies by 1 and 0, so the
    results are bit-identical, which is asserted too."""
    n = 512
    st, tau, push, gz, mu = mixed_states(n, 31)
    tr = horizontal_terrain(mu, n)
    for nsub in (1, 5):
        ref, rflags, rdiag, rstatus = cemu.step(st, tau, push, gz, mu, nsub=nsub)
        got, flags, diag, status = temu.step(st, tau, push, tr, gz, nsub=nsub)
        assert (status == rstatus).all() and (rstatus == 0).all()
        assert (flags == rflags).all()
        for k in STATE + ("foot_force",):
            assert _rel(got[k], ref[k]) <= 1e-14, k
            assert np.array_equal(got[k], ref[k]), k
        assert _rel(diag, rdiag) <= 1e-14 and np.array_equal(diag, rdiag)


def _rot(axis, th):
    return S._rot_axis(np.asarray(axis, dtype=np.float64) / np.linalg.norm(axis), np.array([th]))[0]


@pytest.mark.parametrize("axis,deg", [((1, 0, 0), 90.0), ((0, 1, 0), -90.0), ((0, 0, 1), 37.0), ((1, 2, -0.5), 23.0), ((-0.3, 1, 0.4), 135.0)])
def test_rotating_the_world_changes_nothing(cemu, temu, axis, deg):
    """One rotation R applied to gravity, the base pose and twist, the push and the flat ground (n = R e3, t1 = R e1, t2 = R e2,
    d = ground_z): q, dq, foot_force (sensor frames), flags, status and diag[0..2] equal the flat run's, and position, rotation and
    velocity equal the flat run's rotated by R, to 1e-9 -- a 90 deg roll puts the ground on a wall.  base_rpy is not compared."""
    n = 512
    st, tau, push, gz, mu = mixed_states(n, 32)
    R = _rot(axis, np.deg2rad(deg))
    ref, rflags, rdiag, rstatus = cemu.step(st, tau, push, gz, mu, nsub=3)
    P = util.emu_default_params()
    g = R @ np.array(P.gravity[:])
    P.gravity = (C.c_double * 3)(*g)
    rs = {k: st[k].copy() for k in STATE}
    rs["base_pos"] = R @ st["base_pos"]
    rot = np.einsum("ij,njk->nik", R, st["base_rot"].T.reshape(n, 3, 3))
    rs["base_rot"] = np.ascontiguousarray(rot.reshape(n, 9).T)
    rs["base_rpy"] = np.vstack([np.arctan2(rot[:, 2, 1], rot[:, 2, 2]), np.arctan2(-rot[:, 2, 0], np.hypot(rot[:, 2, 1], rot[:, 2, 2])),
                                np.arctan2(rot[:, 1, 0], rot[:, 0, 0])])
    rs["base_vel"] = np.vstack([R @ st["base_vel"][:3], R @ st["base_vel"][3:]])
    rpush = np.vstack([R @ push[:3], R @ push[3:]])
    tr = np.zeros((40, n))
    for f in range(4):
        tr[10 * f:10 * f + 3] = R[:, 2:3]
        tr[10 * f + 3:10 * f + 6] = R[:, 0:1]
        tr[10 * f + 6:10 * f + 9] = R[:, 1:2]
        tr[10 * f + 9] = mu
    got, flags, diag, status = temu.step(rs, tau, rpush, tr, gz, nsub=3, params=P)
    assert (status == rstatus).all() and (rstatus == 0).all()
    assert (flags == rflags).all()
    for k in ("q", "dq", "foot_force"):
        assert _rel(got[k], ref[k]) <= 1e-9, k
    assert np.abs(diag[:3] - rdiag[:3]).max() <= 1e-9 * max(1.0, np.abs(rdiag[:3]).max())
    # diag[3] counts dual steps: the path, not the result.  Ties at degenerate vertices (an unloaded foot's friction rows meet at
    # one point) break differently under rounding, so a few instances take a step or two more or fewer (measured: 26-36 of 512).
    assert (diag[3] != rdiag[3]).mean() < 0.15 and abs(diag[3].sum() - rdiag[3].sum()) <= 0.01 * rdiag[3].sum()
    assert _rel(got["base_pos"], R @ ref["base_pos"]) <= 1e-9
    assert _rel(got["base_vel"], np.vstack([R @ ref["base_vel"][:3], R @ ref["base_vel"][3:]])) <= 1e-9
    want = np.einsum("ij,njk->nik", R, ref["base_rot"].T.reshape(n, 3, 3)).reshape(n, 9).T
    assert _rel(got["base_rot"], want) <= 1e-9


def tilted_states(n, seed, max_tilt_deg=30.0):
    """mixed_states on per-foot planes: normals up to max_tilt_deg from vertical, tangents at a random in-plane angle, mu per foot in
    [0.05, 1], feet 3 mm into to 4 mm above their planes along the normal.  Returns (st, tau, push, terrain, plane_d)."""
    rng = np.random.default_rng(seed)
    st, tau, push, _, _ = mixed_states(n, seed)
    _, feet = S.forward_kinematics(st["base_pos"], st["base_rot"], st["q"])
    ct = rng.uniform(np.cos(np.deg2rad(max_tilt_deg)), 1.0, (4, n))
    ph = rng.uniform(0.0, 2 * np.pi, (4, n))
    nrm = np.stack([np.sqrt(1 - ct * ct) * np.cos(ph), np.sqrt(1 - ct * ct) * np.sin(ph), ct], axis=1)     # [4, 3, n]
    tr, d = S.terrain_frames(nrm, rng.uniform(0.05, 1.0, (4, n)), feet)
    psi = rng.uniform(0.0, 2 * np.pi, (4, n))
    for f in range(4):
        t1, t2 = tr[10 * f + 3:10 * f + 6].copy(), tr[10 * f + 6:10 * f + 9].copy()
        tr[10 * f + 3:10 * f + 6] = np.cos(psi[f]) * t1 + np.sin(psi[f]) * t2
        tr[10 * f + 6:10 * f + 9] = -np.sin(psi[f]) * t1 + np.cos(psi[f]) * t2
    gap = rng.choice([-0.003, 0.0, 0.001, 0.004], size=(4, n)) * rng.uniform(0.0, 1.0, (4, n))
    gap[rng.uniform(size=(4, n)) < 0.15] = 0.0
    return st, tau, push, tr, d - gap


def test_emulation_matches_the_independent_reference_on_tilted_planes(temu, oracle):
    """512 states on per-foot planes up to 30 deg from horizontal, in groups of one to five substeps: forces within 1e-9, state
    within 1e-10, flags exactly, every kernel-side contact QP's scaled KKT residual <= 1e-10."""
    n = 512
    st, tau, push, tr, d = tilted_states(n, 41)
    nflags = np.zeros(3, int)
    for nsub, idx in enumerate(np.array_split(np.arange(n), 5), start=1):
        sub = {k: np.ascontiguousarray(v[:, idx]) for k, v in st.items()}
        got, flags, diag, status = temu.step(sub, tau[:, idx], push[:, idx], tr[:, idx], d[:, idx], nsub=nsub)
        ref, rflags, _ = CRT.contact_step_terrain(oracle, sub, tau[:, idx], push[:, idx], tr[:, idx], d[:, idx], nsub)
        assert (status == 0).all()
        assert (flags == rflags).all(), np.argwhere(flags != rflags)
        assert np.abs(got["foot_force"] - ref["foot_force"]).max() <= 1e-9 * max(1.0, np.abs(ref["foot_force"]).max()), nsub
        for k in STATE:
            assert np.abs(got[k] - ref[k]).max() <= 1e-10 * max(1.0, np.abs(ref[k]).max()), (nsub, k)
        assert diag[2].max() <= 1e-10, diag[2].max()
        assert diag[1].min() >= 0.0
        nflags += np.bincount(flags.ravel(), minlength=3)
    assert (nflags > 20).all(), nflags


def test_refusals_leave_the_instance_untouched(temu):
    """A non-orthonormal frame or mu < 0 on one foot: WBC_ST_BAD_TERRAIN; a NaN in terrain or plane_d: WBC_ST_NONFINITE.  The
    instance's state and foot_force stay as they were, its flags are 0, and the other instances are those of a clean run."""
    n = 10
    st, tau, push, tr, d = tilted_states(n, 42, max_tilt_deg=10.0)
    st["foot_force"] = np.arange(12 * n, dtype=np.float64).reshape(12, n)
    clean, cflags, cdiag, cstatus = temu.step(st, tau, push, tr, d, nsub=3)
    assert (cstatus == 0).all() and (cflags[:, 2:7] > 0).any()
    bad_tr, bad_d = tr.copy(), d.copy()
    bad_tr[10 * 1 + 0:10 * 1 + 3, 2] *= 1.0 + 1e-8        # foot 1's normal not unit length
    bad_tr[10 * 3 + 3, 3] += 1e-6                           # foot 3's t1 not orthogonal
    bad_tr[10 * 2 + 9, 4] = -0.01                           # mu < 0
    bad_tr[10 * 0 + 7, 5] = np.nan
    bad_d[2, 6] = np.inf
    got, flags, diag, status = temu.step(st, tau, push, bad_tr, bad_d, nsub=3)
    assert list(status[2:7]) == [ST_BAD_TERRAIN] * 3 + [ST_NONFINITE] * 2, status
    ok = np.r_[0:2, 7:n]
    assert (status[ok] == 0).all() and (flags[:, 2:7] == 0).all() and (flags[:, ok] == cflags[:, ok]).all()
    for k in STATE + ("foot_force",):
        assert (got[k][:, 2:7] == st[k][:, 2:7]).all(), k
        assert (got[k][:, ok] == clean[k][:, ok]).all(), k
    # a frame that is orthonormal to within 1e-9 is accepted
    near = tr.copy()
    near[10 * 1 + 0:10 * 1 + 3, 2] *= 1.0 + 2e-10
    assert (temu.step(st, tau, push, near, d, nsub=1)[3] == 0).all()


# --------------------------------------------------------------------------------------------------- CPU: closed loop, emulation
def _closed_loop_terrain(emu, temu, sc, tr, d, cycles, ctrl_terrain, each=None):
    """The controller (host emulation of wbc_cycle, observer off; terrain = ctrl_terrain) closed through the terrain plant."""
    n = sc["q"].shape[1]
    P = util.emu_default_params()
    P.observer_enabled = 0
    sc["terrain"] = ctrl_terrain
    for c in range(cycles):
        res = emu.cycle(sc, params=P)
        assert (res["status"] == 0).all()
        before = {k: sc[k].copy() for k in STATE}
        out = temu.step(sc, res["tau"], np.zeros((6, n)), tr, d, nsub=5)
        assert (out[3] == 0).all()
        for k in STATE + ("foot_force",):
            sc[k] = out[0][k]
        if each:
            each(c, before, out, res)
    return sc


def test_stick_on_a_15_degree_slope(emu, temu):
    """mu = 0.6 > tan 15 deg, the controller given the slope's frames: all four feet stick on every cycle for 1 s and drift less
    than 0.1 mm."""
    n = 2
    sc, _ = _standing(n, 61)
    _, feet0 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    tr, d = S.slope_terrain(feet0, np.deg2rad(15.0), np.array([0.0, 2.2]), 0.6)
    seen = []
    sc = _closed_loop_terrain(emu, temu, sc, tr, d, 400, tr, each=lambda c, b, out, res: seen.append(out[1].copy()))
    assert (np.array(seen) == 1).all()
    _, feet1 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    drift = np.abs(feet1 - feet0).max()
    assert drift < 1e-4, drift
    print("stick on a 15 deg slope: foot drift %.2e m over 1 s" % drift)


def test_slip_on_a_15_degree_slope(emu, temu, oracle):
    """mu = 0.1 < tan 15 deg: the feet slide (flag 2) and the base moves downhill.  In each sliding foot's frame, the tangential
    impulse lies on the pyramid's boundary, friction does no positive work, and the velocity along n after the step stays within the
    relaxation's bound target + mu (|v_t1| + |v_t2|) -- test_slip of the flat plant, in the foot's frame."""
    n, mu, az = 2, 0.1, np.array([0.0, 2.2])
    sc, _ = _standing(n, 62)
    _, feet0 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    tr, d = S.slope_terrain(feet0, np.deg2rad(15.0), az, mu)
    sc["terrain"] = tr
    P = util.emu_default_params()
    P.observer_enabled = 0
    pos0 = sc["base_pos"].copy()
    slides = 0
    for c in range(40):
        res = emu.cycle(sc, params=P)
        st = {k: sc[k] for k in STATE}
        ref, rflags, lam = CRT.contact_step_terrain(oracle, st, res["tau"], np.zeros((6, n)), tr, d, 1)
        got, flags, diag, status = temu.step(st, res["tau"], np.zeros((6, n)), tr, d, nsub=1)
        assert (status == 0).all() and (flags == rflags).all()
        for i in range(n):
            one = {k: st[k][:, i:i + 1] for k in STATE}
            one.update({k: np.zeros((m, 1)) for k, m in CR._ZERO_FIELDS.items()})
            one["mode"] = np.zeros(1, np.int32)
            dd = oracle.update_only(one, 0)
            J = np.array(dd.Jac_lin).reshape(12, 18)
            v = J @ np.concatenate([got["base_vel"][:, i], got["dq"][:, i]])
            fp = np.array(dd.foot_pos).reshape(4, 3)
            for k in range(4):
                if flags[k, i] != 2:
                    continue
                slides += 1
                F = np.column_stack([tr[10 * k + 3:10 * k + 6, i], tr[10 * k + 6:10 * k + 9, i], tr[10 * k:10 * k + 3, i]])
                vk = F.T @ v[3 * k:3 * k + 3]
                lk = lam[3 * k:3 * k + 3, i]
                phi = F[:, 2] @ fp[k] - d[k, i]
                assert min(abs(abs(lk[0]) - mu * lk[2]), abs(abs(lk[1]) - mu * lk[2])) <= 1e-9 * lk[2]
                assert lk[0] * vk[0] + lk[1] * vk[1] <= 1e-12 * np.abs(lk).max()
                target = -(1.0 if phi >= 0 else 0.2) * phi / 0.0025
                assert vk[2] - target <= mu * (abs(vk[0]) + abs(vk[1])) * (1 + 1e-6) + 1e-9
        for k in STATE + ("foot_force",):
            sc[k] = got[k]
    downhill = (sc["base_pos"][0] - pos0[0]) * np.cos(az) + (sc["base_pos"][1] - pos0[1]) * np.sin(az)
    assert slides > 40, slides
    assert (downhill > 1e-3).all(), downhill
    print("slip on a 15 deg slope: %d sliding foot-steps, base %.1f mm downhill in 0.1 s" % (slides, 1e3 * downhill.min()))


def groove_terrain(feet, deg, mu):
    """A V-groove along the robot's y axis: the left feet (BL, FL; x < 0) on a plane falling toward +x, the right feet (BR, FR) on
    one falling toward -x, each at `deg` from horizontal, through the feet's current points."""
    n = feet.shape[0]
    s, c = np.sin(np.deg2rad(deg)), np.cos(np.deg2rad(deg))
    nrm = np.zeros((4, 3, n))
    for f, side in enumerate((-1.0, 1.0, 1.0, -1.0)):       # stacked BR, BL, FL, FR: the normal leans toward the groove's middle
        nrm[f] = np.array([side * s, 0.0, c])[:, None]
    return S.terrain_frames(nrm, mu, feet)


def test_the_controllers_terrain_input_matters(emu, temu):
    """A V-groove of two 25 deg planes at mu = 0.3 < tan 25 deg (0.47).  Given the groove's frames (with mu = 0.25, a margin below
    the ground's), the controller stands by pushing along the normals: every foot sticks on every cycle for 1 s.  Given
    terrain = NULL, it plans vertical forces, which lie outside the real cones, and the feet slide.
    Measured on the emulation (seed 63, two robots): with the frames, foot drift 1.4e-9 m over 1 s and no sliding foot-cycle;
    without them, 66 % sliding foot-cycles from the first cycle on and 0.53 m of foot drift in 0.25 s (the robots fall into the
    groove).  Told the ground's own mu = 0.3, the controller plans forces on the cone's edge: the plant then flags 44 % of the
    foot-cycles as sliding (a friction row active), with 16 um of drift over 1 s."""
    n = 2
    sc, _ = _standing(n, 63)
    _, feet0 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    tr, d = groove_terrain(feet0, 25.0, 0.3)
    told, _ = groove_terrain(feet0, 25.0, 0.25)
    flags = []
    a = _closed_loop_terrain(emu, temu, {k: v.copy() for k, v in sc.items()}, tr, d, 400, told,
                             each=lambda c, b, out, res: flags.append(out[1].copy()))
    _, feet1 = S.forward_kinematics(a["base_pos"], a["base_rot"], a["q"])
    drift_with = np.abs(feet1 - feet0).max()
    assert (np.array(flags) == 1).all()
    assert drift_with < 1e-6, drift_with
    flags2 = []
    b = _closed_loop_terrain(emu, temu, {k: v.copy() for k, v in sc.items()}, tr, d, 100, None,
                             each=lambda c, b_, out, res: flags2.append(out[1].copy()))
    _, feet2 = S.forward_kinematics(b["base_pos"], b["base_rot"], b["q"])
    drift_without = np.abs(feet2 - feet0).max()
    slid = (np.array(flags2) == 2).mean()
    assert (np.array(flags2[:5]) == 2).any()
    assert slid > 0.3, slid
    assert drift_without > 0.05, drift_without
    print("V-groove 25 deg, mu 0.3: with the frames drift %.1e m over 1 s; without them %.0f %% sliding foot-cycles, drift %.0f mm in 0.25 s"
          % (drift_with, 100 * slid, 1e3 * drift_without))


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_matches_emulation_host_and_device_pointers(gpu_batch, temu, cemu):
    import torch
    n = 4096
    st, tau, push, tr, d = tilted_states(n, 71)
    ref, rflags, rdiag, rstatus = temu.step(st, tau, push, tr, d, nsub=5)
    assert (rstatus == 0).all()
    h = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
    h["foot_force"] = np.zeros((12, n))
    contact, diag, status = np.zeros((4, n), np.int32), np.zeros((4, n)), np.full(n, 7, np.int32)
    gpu_batch.plant_contact_step(h, tau, push, terrain=tr, plane_d=d, substeps=5, contact=contact, diag=diag, status=status)
    assert gpu_batch.last_launches() == 1
    dev = torch.device("cuda", 0)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dd_ = {k: T(st[k]) for k in STATE}
    dd_["foot_force"] = torch.zeros(12, n, dtype=torch.float64, device=dev)
    dc, dd, ds = torch.zeros(4, n, dtype=torch.int32, device=dev), torch.zeros(4, n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)
    gpu_batch.plant_contact_step(dd_, T(tau), T(push), terrain=T(tr), plane_d=T(d), substeps=5, contact=dc, diag=dd, status=ds)
    for got, c, dg, s in ((h, contact, diag, status), ({k: v.cpu().numpy() for k, v in dd_.items()}, dc.cpu().numpy(), dd.cpu().numpy(), ds.cpu().numpy())):
        assert (s == 0).all() and (c == rflags).all()
        for k in STATE + ("foot_force",):
            assert np.abs(got[k] - ref[k]).max() <= 1e-10 * max(1.0, np.abs(ref[k]).max()), k
        assert dg[2].max() <= 1e-10 and np.abs(dg[0] - rdiag[0]).max() <= 1e-12
    # horizontal terrain through the new entry point equals wbc_plant_contact_step's output
    st2, tau2, push2, gz2, mu2 = mixed_states(n, 72)
    outs = []
    for kw in (dict(ground_z=gz2, mu=mu2), dict(terrain=horizontal_terrain(mu2, n), plane_d=gz2)):
        h2 = {k: np.array(st2[k], dtype=np.float64, order="C") for k in STATE}
        h2["foot_force"] = np.zeros((12, n))
        c2, d2, s2 = np.zeros((4, n), np.int32), np.zeros((4, n)), np.full(n, 7, np.int32)
        gpu_batch.plant_contact_step(h2, tau2, push2, substeps=5, contact=c2, diag=d2, status=s2, **kw)
        outs.append((h2, c2, d2, s2))
    (a, ca, da, sa), (b, cb, db, sb) = outs
    assert (sa == 0).all() and (sa == sb).all() and (ca == cb).all()
    for k in STATE + ("foot_force",):
        assert _rel(b[k], a[k]) <= 1e-14, k
    assert _rel(db, da) <= 1e-14
    # refusals on the device: a bad frame and a NaN offset
    tr3, d3 = tr.copy(), d.copy()
    tr3[10 * 2 + 9, 5] = -1.0
    d3[1, 9] = np.nan
    h3 = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
    h3["foot_force"] = np.zeros((12, n))
    s3 = np.zeros(n, np.int32)
    gpu_batch.plant_contact_step(h3, tau, push, terrain=tr3, plane_d=d3, substeps=5, status=s3)
    assert s3[5] == ST_BAD_TERRAIN and s3[9] == ST_NONFINITE and (np.delete(s3, [5, 9]) == 0).all()
    assert (h3["q"][:, [5, 9]] == st["q"][:, [5, 9]]).all()


@pytest.mark.gpu
def test_closed_loop_trot_on_slopes_through_the_terrain_plant(gpu_batch):
    """4096 robots, each on its own slope of up to 10 deg (random downhill azimuth) at mu = 0.6, trotting in place with
    test_contact_plant's schedule (swings end at touchdown or the phase end), closed for 320 cycles through the terrain plant; the
    controller gets the same terrain.  No solve fails, no normal force is negative, no foot sinks 2 mm along its normal, every swing
    foot is airborne at mid-swing, and the robots stay up.  First run on a B200: 0 failed solves, smallest normal force 0 N,
    penetration below 1 um, 32 768 / 32 768 swing feet airborne at mid-swing, every robot-swing ended by touchdown, max |base drift|
    7.3 mm and max |rpy - rpy0| 0.020 rad; the bounds below are 30 mm and 0.1 rad."""
    import torch
    from tests.test_fdyn_plant import trot_in_place_targets
    n, P, height = 4096, 40, 0.03
    sched = [S.MODE_STANCE, S.MODE_SWING_BR_FL, S.MODE_STANCE, S.MODE_SWING_BL_FR]
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=44)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    rng = np.random.default_rng(12)
    tr, d = S.slope_terrain(feet, np.deg2rad(rng.uniform(0.0, 10.0, n)), rng.uniform(0.0, 2 * np.pi, n), 0.6)
    sc["terrain"] = tr
    nrm = np.stack([tr[10 * f:10 * f + 3] for f in range(4)])          # [4, 3, n]
    base0 = sc["base_pos"].copy()
    dev = torch.device("cuda", 0)
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    zero = torch.zeros(6, n, dtype=torch.float64, device=dev)
    dtr, dd = din["terrain"], torch.from_numpy(d).to(dev)
    contact = torch.zeros(4, n, dtype=torch.int32, device=dev)
    diag = torch.zeros(4, n, dtype=torch.float64, device=dev)
    cstatus = torch.zeros(n, dtype=torch.int32, device=dev)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    fails, cfails, fzmin, pen, slips, touchdowns, airborne_mid, mid_checks = 0, 0, 1e9, 0.0, 0, 0, 0, 0
    anchor, landed = None, None
    for c in range(8 * P):
        mode = sched[(c // P) % 4]
        s = (c % P) / P
        first, second = (1, 3) if mode == S.MODE_SWING_BL_FR else (0, 2)
        if c % P == 0:
            host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
            _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
            landed = np.zeros(n, bool)
        if mode != S.MODE_STANCE:
            cf = contact.cpu().numpy()
            td = (~landed) & (s > 0.5) & (cf[first] > 0) & (cf[second] > 0)
            touchdowns += int(td.sum())
            landed |= td
            m = np.where(landed, S.MODE_STANCE, mode).astype(np.int32)
        else:
            m = np.full(n, mode, np.int32)
        din["mode"] = torch.from_numpy(m).to(dev)
        sp, sv, sa = trot_in_place_targets(anchor, mode, s, P * 0.0025, height)
        din["sw_des_pos"].copy_(torch.from_numpy(sp)); din["sw_des_vel"].copy_(torch.from_numpy(sv)); din["sw_des_acc"].copy_(torch.from_numpy(sa))
        gpu_batch.cycle_device(din, dout, n, n)
        fails += int((dout["status"] != 0).sum().item())
        gpu_batch.plant_contact_step(din, dout["tau"], zero, terrain=dtr, plane_d=dd, n=n, ld=n, substeps=5, contact=contact, diag=diag,
                                     status=cstatus)
        cfails += int((cstatus != 0).sum().item())
        dg = diag.cpu().numpy()
        fzmin = min(fzmin, float(dg[1].min()))
        pen = max(pen, float(dg[0].max()))
        cf = contact.cpu().numpy()
        slips += int((cf == 2).sum())
        if mode != S.MODE_STANCE and c % P == P // 2:
            mid_checks += 2 * n
            airborne_mid += int((cf[first] == 0).sum() + (cf[second] == 0).sum())
    host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q", "base_rpy")}
    _, ft = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
    final_pen = max(0.0, float((d - np.einsum("fkn,nfk->fn", nrm, ft)).max()))
    drift = np.abs(host["base_pos"] - base0).max()
    datt = np.abs(host["base_rpy"] - sc["base_rpy"]).max()
    print("closed-loop trot on slopes through the terrain plant: %d robots x %d cycles, failed solves %d / %d, min normal force %.3f N, "
          "max penetration %.3f mm (final %.3f mm), swing feet airborne at mid-swing %d / %d, %d sliding foot-cycles, %d touchdowns "
          "before the phase end, max |base drift| %.1f mm, max |rpy - rpy0| %.3f rad"
          % (n, 8 * P, fails, cfails, fzmin, 1e3 * pen, 1e3 * final_pen, airborne_mid, mid_checks, slips, touchdowns, 1e3 * drift, datt))
    assert fails == 0 and cfails == 0
    assert fzmin >= 0.0 and pen < 2e-3 and final_pen < 2e-3
    assert airborne_mid == mid_checks
    assert drift < 0.03 and datt < 0.1
