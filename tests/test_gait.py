"""The trot gait generator (wbc_gait_init / wbc_gait_step, csrc/wbc_gait.cuh).

CPU: the kernel's source compiled for the host (tests/host_emu/gait_emu.cpp) against an independent numpy restatement of the law
(tests/gait_ref.py); the swing curve and CoM reference against their own derivatives; the schedule, touchdown, leash and refusals;
and the controller, the contact plant and the gait closed on the CPU, walking to forward, backward, lateral and turning commands.
GPU: the kernels against the emulation with host and device pointers, and herds of 4096 robots walking to per-robot commands through
gait_step -> cycle_device -> plant_contact_step on one stream, on flat ground and on a slope per robot."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import gait_ref as GR
from tests import util
from tests.test_contact_plant import ContactEmu
from wbc_quadruped_dob_b200 import scenarios as S

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
STATE = ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")
GS_INT = ("phase", "tick", "landed")
GS_DBL = ("com_ref", "v_ref", "liftoff", "target", "offset")
DT = 0.0025
DEFAULTS = dict(stance_cycles=46, swing_cycles=46, step_height=0.03, k_v=0.1, max_step=0.1, acc_lin=1.0, acc_yaw=2.0, leash=0.05)
DCOM = 2.0 * np.sqrt(2500.0 * S.TOTAL_MASS)     # critically damped CoM gains, as test_contact_plant.py's closed loops


class _GaitParams(C.Structure):
    _fields_ = [("ns", C.c_int), ("nw", C.c_int)] + [(k, C.c_double) for k in ("step_height", "k_v", "max_step", "acc_lin", "acc_yaw", "leash")]


class _GaitIO(C.Structure):
    _fields_ = [(k, _dp) for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "cmd")] + [("contact", _ip), ("terrain", _dp),
                ("plane_d", _dp), ("k0", _ip), ("phase", _ip), ("tick", _ip), ("landed", _ip)] + [(k, _dp) for k in GS_DBL] + \
               [("mode", _ip), ("des", _dp * 6), ("out_ld", C.c_long), ("status", _ip), ("ld", C.c_long)]


def _gp(**kw):
    g = dict(DEFAULTS, **kw)
    return g, _GaitParams(g["stance_cycles"], g["swing_cycles"], *[g[k] for k in ("step_height", "k_v", "max_step", "acc_lin", "acc_yaw", "leash")])


class GaitEmu:
    """g++ build of gait_init_instance / gait_step_instance (test infrastructure only)."""

    def __init__(self):
        so = os.path.join(util.EMU_DIR, "libgait_emu.so")
        util._build_emu(os.path.join(util.EMU_DIR, "gait_emu.cpp"), so)
        self.lib = C.CDLL(so)
        for f in (self.lib.emu_gait_init, self.lib.emu_gait_step):
            f.argtypes = [C.POINTER(_GaitParams), C.c_double, C.POINTER(_GaitIO), C.c_int]
            f.restype = None

    @staticmethod
    def _io(st, gs, n, keep, cmd=None, contact=None, terrain=None, plane_d=None, k0=None, out=None, status=None):
        io = _GaitIO()
        d = lambda a: None if a is None else a.ctypes.data_as(_dp)
        i = lambda a: None if a is None else a.ctypes.data_as(_ip)
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q"):
            a = np.ascontiguousarray(st[k], dtype=np.float64); keep.append(a); setattr(io, k, d(a))
        for name, a, conv in (("cmd", cmd, np.float64), ("terrain", terrain, np.float64), ("plane_d", plane_d, np.float64),
                              ("contact", contact, np.int32), ("k0", k0, np.int32)):
            if a is not None:
                a = np.ascontiguousarray(a, dtype=conv); keep.append(a)
            setattr(io, name, (d if conv is np.float64 else i)(a))
        for k in GS_INT:
            setattr(io, k, i(gs[k]))
        for k in GS_DBL:
            setattr(io, k, d(gs[k]))
        if out is not None:
            io.mode = i(out["mode"])
            for b, k in enumerate(GR.OUT):
                io.des[b] = d(out[k])
        io.out_ld = n; io.ld = n
        io.status = i(status)
        return io

    def init(self, G, st, k0=None, terrain=None, plane_d=None, gs=None):
        n = st["q"].shape[1]
        gs = gs or {**{k: np.zeros((1, n), np.int32) for k in GS_INT}, **{k: np.zeros((m, n)) for k, m in zip(GS_DBL, (4, 3, 6, 6, 8))}}
        status, keep = np.full(n, 7, np.int32), []
        io = self._io(st, gs, n, keep, terrain=terrain, plane_d=plane_d, k0=k0, status=status)
        self.lib.emu_gait_init(C.byref(_gp(**G)[1]), DT, C.byref(io), n)
        return gs, status

    def step(self, G, gs, st, cmd=None, contact=None, terrain=None, plane_d=None, out=None):
        """Advances gs in place; returns (outputs, status)."""
        n = st["q"].shape[1]
        out = out or {"mode": np.zeros(n, np.int32), **{k: np.zeros((6, n)) for k in GR.OUT}}
        status, keep = np.full(n, 7, np.int32), []
        io = self._io(st, gs, n, keep, cmd=cmd, contact=contact, terrain=terrain, plane_d=plane_d, out=out, status=status)
        self.lib.emu_gait_step(C.byref(_gp(**G)[1]), DT, C.byref(io), n)
        return out, status


@pytest.fixture(scope="module")
def gemu():
    return GaitEmu()


def _copy(gs):
    return {k: v.copy() for k, v in gs.items()}


def _rot(rpy):
    return np.ascontiguousarray(S.rpy_to_rot(rpy).reshape(rpy.shape[1], 9).T)


class Drift:
    """Random robot states that wander: the base drifts at a per-robot velocity plus noise, yaw turns, joints jitter."""

    def __init__(self, n, seed):
        self.rng = np.random.default_rng(seed)
        sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), seed=seed)
        self.st = {k: np.ascontiguousarray(sc[k]) for k in STATE}
        self.v = self.rng.uniform(-0.3, 0.3, (3, n)) * np.array([[1.0], [0.5], [0.0]])
        self.w = self.rng.uniform(-0.5, 0.5, n)

    def next(self):
        st, rng, n = self.st, self.rng, self.st["q"].shape[1]
        st["base_pos"] = st["base_pos"] + self.v * DT + rng.normal(0.0, 5e-4, (3, n))
        st["base_vel"] = np.vstack([self.v + rng.normal(0.0, 0.05, (3, n)), rng.normal(0.0, 0.1, (3, n))])
        st["base_rpy"] = st["base_rpy"] + np.vstack([rng.normal(0.0, 1e-3, (2, n)), self.w * DT])
        st["base_rot"] = _rot(st["base_rpy"])
        st["q"] = np.clip(st["q"] + rng.normal(0.0, 2e-3, (12, n)), S.QMIN[:, None], S.QMAX[:, None])
        return st


def _assert_same(got, ref, what, tol=1e-12):
    for k, r in ref.items():
        g = got[k]
        if r.dtype.kind == "i":
            assert (g == r).all(), (what, k, np.argwhere(g != r)[:5])
        else:
            err = np.abs(g - r).max() / max(1.0, np.abs(r).max())
            assert err <= tol, (what, k, err)


def _slope(n, seed, feet, max_deg=15.0):
    rng = np.random.default_rng(seed)
    return S.slope_terrain(feet, np.deg2rad(rng.uniform(0.0, max_deg, n)), rng.uniform(0.0, 2 * np.pi, n), 0.6)


@pytest.mark.parametrize("ground", ["flat", "slope"])
def test_emulation_matches_the_independent_reference(gemu, ground):
    """256 robots x 400 cycles per ground: random wandering states, per-robot commands that change every 100 cycles, random start
    offsets and contact flags.  Integer state and mode equal, doubles to 1e-12."""
    n, cycles = 256, 400
    rng = np.random.default_rng(31 if ground == "flat" else 32)
    G = DEFAULTS if ground == "flat" else dict(DEFAULTS, stance_cycles=30, swing_cycles=24, k_v=0.2, max_step=0.04, acc_lin=0.5, leash=0.02)
    drift = Drift(n, 33 if ground == "flat" else 34)
    st = drift.st
    terrain = plane_d = None
    if ground == "slope":
        _, _, feet = GR.kinematics(st)
        terrain, plane_d = _slope(n, 35, feet)
    k0 = rng.integers(-50, 400, n).astype(np.int32)
    gs, status = gemu.init(G, st, k0, terrain, plane_d)
    rgs, rstatus = GR.init(G, DT, st, k0, terrain, plane_d)
    assert (status == 0).all() and (rstatus == 0).all()
    _assert_same(gs, rgs, "init")
    landed = swings_clamped = 0
    for c in range(cycles):
        if c % 100 == 0:
            cmd = np.vstack([rng.uniform(-0.4, 0.4, n), rng.uniform(-0.2, 0.2, n), rng.uniform(-0.6, 0.6, n)])
        contact = (rng.uniform(size=(4, n)) < 0.4) * rng.integers(1, 3, (4, n))
        st = drift.next()
        out, status = gemu.step(G, gs, st, cmd, contact, terrain, plane_d)
        rgs, rout, rstatus = GR.step(G, DT, rgs, st, cmd, contact, terrain, plane_d)
        assert (status == 0).all() and (rstatus == 0).all()
        _assert_same(gs, rgs, "state, cycle %d" % c)
        _assert_same(out, rout, "outputs, cycle %d" % c)
        landed += int(gs["landed"].sum())
        swings_clamped += int((np.abs(rout["com_des_pos"][0:2] - GR.kinematics(st)[0][:, 0:2].T).max(axis=0) > 0.99 * G["leash"]).sum())
    assert landed > 0 and swings_clamped > 0          # touchdowns and the leash both occur


def _steady(n=4, seed=41):
    """Standing robots (zero velocity), the state the gait is held on in the property tests."""
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), seed=seed)
    st = {k: np.ascontiguousarray(sc[k]) for k in STATE}
    st["base_vel"] = np.zeros((6, n))
    return st


def test_swing_curve_and_com_reference_are_consistent(gemu):
    """At the touchdown tick the swing foot is at p1 with zero velocity and zero horizontal acceleration (the quintic's); the lift
    profile's vertical acceleration there is 2 pi^2 h / T^2 (sin^2 has no zero-acceleration ends).  At the lift-off tick the foot is
    within the curve's first step of p0.  Central differences over ticks of sw_des_pos and com_des_pos match the emitted velocities
    and accelerations to the differences' truncation error; the CoM reference is followed under a ramping, turning command."""
    n, G = 4, dict(DEFAULTS, leash=10.0)
    st = _steady(n)
    gs, _ = gemu.init(G, st, np.full(n, 45, np.int32))        # lift-off at the next step
    cmd = np.vstack([np.full(n, 0.3), np.full(n, -0.1), np.full(n, 0.5)])
    outs = []
    for c in range(1 + 46):
        out, status = gemu.step(G, gs, st, cmd)
        assert (status == 0).all()
        outs.append({k: v.copy() for k, v in out.items()})
    lift, td = outs[1], outs[46]
    p0, p1 = gs["liftoff"], gs["target"]
    h, T, Nw = G["step_height"], 46 * DT, 46
    assert np.abs(td["sw_des_pos"] - p1).max() < 1e-12
    assert np.abs(td["sw_des_vel"]).max() < 1e-12
    acc = td["sw_des_acc"]
    assert np.abs(acc[[0, 1, 3, 4]]).max() < 1e-9 and np.abs(acc[[2, 5]] - 2 * np.pi ** 2 * h / T ** 2).max() < 1e-9
    s0 = 1.0 / Nw
    sig0 = 10 * s0 ** 3 - 15 * s0 ** 4 + 6 * s0 ** 5
    step0 = np.abs(p1 - p0).max() * sig0 + h * np.sin(np.pi * s0) ** 2
    assert np.abs(lift["sw_des_pos"] - p0).max() <= step0 + 1e-12
    P = np.array([o["sw_des_pos"] for o in outs[1:]]); V = np.array([o["sw_des_vel"] for o in outs[1:]]); A = np.array([o["sw_des_acc"] for o in outs[1:]])
    dP = (P[2:] - P[:-2]) / (2 * DT)
    dV = (V[2:] - V[:-2]) / (2 * DT)
    assert np.abs(dP - V[1:-1]).max() < 5e-3 * np.abs(V).max(), np.abs(dP - V[1:-1]).max()
    assert np.abs(dV - A[1:-1]).max() < 5e-3 * np.abs(A).max(), np.abs(dV - A[1:-1]).max()
    # CoM (semi-implicit: each step moves the reference by the new velocity): backward differences of the position are the emitted
    # velocity; those of the velocity are the emitted acceleration up to the first-order terms of the rotation over one step,
    # (omega |a| + omega^2 |v|) dt
    CP = np.array([o["com_des_pos"] for o in outs]); CV = np.array([o["com_des_vel"] for o in outs]); CA = np.array([o["com_des_acc"] for o in outs])
    rows = [0, 1, 5]
    assert np.abs((CP[1:, rows] - CP[:-1, rows]) / DT - CV[1:, rows]).max() < 1e-9
    assert np.abs((CV[1:, rows] - CV[:-1, rows]) / DT - CA[1:, rows]).max() < (0.5 * G["acc_lin"] + 0.5 ** 2 * 0.32) * DT
    ramp = np.minimum(0.5, G["acc_yaw"] * DT * np.arange(1, len(outs) + 1))[:, None]          # the yaw rate ramps toward 0.5
    assert np.abs(CV[:, 5] - ramp).max() < 1e-12 and np.abs(CA[:, 5] - G["acc_yaw"]).max() < 1e-9
    assert (CP[:, 2] == CP[0, 2]).all() and (CV[:, 2] == 0).all()


def test_schedule_touchdown_and_leash(gemu):
    """contact = NULL: the modes are exactly the phase schedule.  Flags before s > 0.5 do not end a swing; flags after it end it on that
    cycle (the mode is stance from then on, to the phase end).  The CoM reference stays within the leash of the measured CoM."""
    n, G = 3, dict(DEFAULTS, stance_cycles=5, swing_cycles=8, leash=0.01)
    st = _steady(n)
    gs, _ = gemu.init(G, st, np.array([0, 3, 9], np.int32))
    sched = [S.MODE_STANCE] * 5 + [S.MODE_SWING_BR_FL] * 8 + [S.MODE_STANCE] * 5 + [S.MODE_SWING_BL_FR] * 8
    cmd = np.vstack([np.full(n, 1.0), np.zeros(n), np.zeros(n)])
    _, _, feet = GR.kinematics(st)
    for c in range(3 * 26):
        out, _ = gemu.step(G, gs, st, cmd)
        assert [int(m) for m in out["mode"]] == [sched[(c + k) % 26] for k in (0, 3, 9)]
        e = out["com_des_pos"][0:2] - GR.kinematics(st)[0][:, 0:2].T
        assert np.sqrt((e ** 2).sum(axis=0)).max() <= 0.01 * (1 + 1e-12)
    # touchdown: robot 0 enters swing{BR,FL} at its 5th step; flags on from its first swing tick
    gs, _ = gemu.init(G, st, np.zeros(n, np.int32))
    contact = np.ones((4, n), np.int32)
    modes = []
    for c in range(26):
        out, _ = gemu.step(G, gs, st, None, contact)
        modes.append(int(out["mode"][0]))
    # s = (tick + 1) / 8 > 0.5 first at tick 4: ticks 0..3 swing, then stance to the phase end
    assert modes[5:13] == [S.MODE_SWING_BR_FL] * 4 + [S.MODE_STANCE] * 4, modes
    assert modes[18:26] == [S.MODE_SWING_BL_FR] * 4 + [S.MODE_STANCE] * 4, modes
    # flags only before mid-swing: the swing lasts its phase
    gs, _ = gemu.init(G, st, np.zeros(n, np.int32))
    modes = []
    for c in range(13):
        out, _ = gemu.step(G, gs, st, None, contact if 5 <= c < 9 else np.zeros((4, n), np.int32))
        modes.append(int(out["mode"][0]))
    assert modes[5:13] == [S.MODE_SWING_BR_FL] * 8, modes
    # one swing foot down is not a touchdown
    gs, _ = gemu.init(G, st, np.zeros(n, np.int32))
    one = np.zeros((4, n), np.int32); one[0] = 1
    modes = [int(gemu.step(G, gs, st, None, one)[0]["mode"][0]) for c in range(13)]
    assert modes[5:13] == [S.MODE_SWING_BR_FL] * 8, modes


def test_refusals_leave_state_and_outputs_untouched(gemu):
    """Non-finite inputs and bad terrain frames are refused per robot with nothing written; a corrupt phase or tick is refused with
    WBC_ST_BAD_MODE."""
    n = 6
    st = _steady(n)
    _, _, feet = GR.kinematics(st)
    terrain, plane_d = _slope(n, 3, feet, 10.0)
    gs, status = gemu.init(DEFAULTS, st, None, terrain, plane_d)
    assert (status == 0).all()
    bad_st = {k: v.copy() for k, v in st.items()}
    bad_st["q"][4, 1] = np.nan
    bad_t = terrain.copy()
    bad_t[3, 2] += 1e-6                                  # t1 of foot 0 no longer unit
    bad_t[10 * 2 + 0:10 * 2 + 3, 3] = [0.0, np.sin(1.1), np.cos(1.1)]     # a normal 63 deg from vertical (n_z < 0.5)
    gs["phase"][0, 4] = 5
    gs["com_ref"][0, 5] = np.inf
    before = _copy(gs)
    out = {"mode": np.full(n, 9, np.int32), **{k: np.full((6, n), 7.0) for k in GR.OUT}}
    out, status = gemu.step(DEFAULTS, gs, bad_st, None, None, bad_t, plane_d, out=out)
    assert list(status) == [0, GR.ST_NONFINITE, GR.ST_BAD_TERRAIN, GR.ST_BAD_TERRAIN, GR.ST_BAD_MODE, GR.ST_NONFINITE], status
    for i in range(1, 6):
        assert out["mode"][i] == 9 and all((out[k][:, i] == 7.0).all() for k in GR.OUT)
        assert all((gs[k][:, i] == before[k][:, i]).all() for k in gs)
    assert out["mode"][0] != 9 and gs["tick"][0, 0] == before["tick"][0, 0] + 1
    gs2, status = gemu.init(DEFAULTS, bad_st, None, bad_t, plane_d, gs=_copy(before))
    assert list(status[:4]) == [0, GR.ST_NONFINITE, GR.ST_BAD_TERRAIN, GR.ST_BAD_TERRAIN]
    for i in (1, 2, 3):
        assert all((gs2[k][:, i] == before[k][:, i]).all() for k in gs2)


# ---------------------------------------------------------------------------------------------------------- closed loop
def _standing(n, seed):
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=seed)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    sc["base_rpy"] = np.vstack([np.zeros((2, n)), sc["base_rpy"][2]])       # level, at a random heading, in the nominal stand
    sc["base_rot"] = _rot(sc["base_rpy"])
    sc["q"] = np.repeat(S.Q_NOMINAL[:, None], n, axis=1)
    com, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["sw_des_pos"] = np.zeros((6, n)); sc["sw_des_vel"] = np.zeros((6, n)); sc["sw_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    sc["obs_yd"] = np.zeros((6, n)); sc["obs_yw"] = np.zeros((6, n))
    return sc, feet


def walk_on_cpu(emu, cemu, gemu, cmd, cycles, seed=61, G=DEFAULTS, k0=None):
    """The controller (host emulation of wbc_cycle, observer off, critically damped CoM gains), the contact plant (flat ground at the
    feet's start height 0 after a shift) and the gait, closed for `cycles` cycles.  Returns per-cycle records."""
    n = cmd.shape[1]
    sc, feet = _standing(n, seed)
    # put the ground at z = 0 under the lowest foot: the gait's flat ground is z = 0
    sc["base_pos"] = sc["base_pos"] - np.array([[0.0], [0.0], [1.0]]) * feet[:, :, 2].min(axis=1)[None]
    _, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    gz = np.zeros((4, n))
    P = util.emu_default_params()
    P.observer_enabled = 0
    P.dcom = DCOM
    gs, status = gemu.init(G, sc, k0)
    assert (status == 0).all()
    contact = np.zeros((4, n), np.int32)
    rec = {"vel": [], "rpy": [], "z": [], "fzmin": [], "pen": [], "mode": []}
    for c in range(cycles):
        out, status = gemu.step(G, gs, sc, cmd, contact)
        assert (status == 0).all()
        sc["mode"] = out["mode"]
        for k in GR.OUT:
            sc[k] = out[k]
        res = emu.cycle(sc, params=P)
        assert (res["status"] == 0).all(), (c, res["status"])
        nxt, contact, diag, cstatus = cemu.step({k: sc[k] for k in STATE + ("foot_force",)}, res["tau"], np.zeros((6, n)), gz, np.full(n, 0.6))
        assert (cstatus == 0).all()
        for k in STATE + ("foot_force",):
            sc[k] = nxt[k]
        R = sc["base_rot"].T.reshape(n, 3, 3)
        yaw = sc["base_rpy"][2]
        v = sc["base_vel"][0:2]
        rec["vel"].append(np.vstack([np.cos(yaw) * v[0] + np.sin(yaw) * v[1], -np.sin(yaw) * v[0] + np.cos(yaw) * v[1], sc["base_vel"][5]]))
        rec["rpy"].append(sc["base_rpy"].copy()); rec["z"].append(sc["base_pos"][2].copy())
        rec["fzmin"].append(diag[1].min()); rec["pen"].append(diag[0].max()); rec["mode"].append(out["mode"].copy())
    return {k: np.array(v) for k, v in rec.items()}


COMMANDS = np.array([[0.2, 0.0, 0.0], [-0.2, 0.0, 0.0], [0.0, 0.1, 0.0], [0.0, -0.1, 0.0], [0.0, 0.0, 0.4], [0.0, 0.0, -0.4],
                     [0.15, 0.05, 0.2], [0.0, 0.0, 0.0]]).T


def tracking(rec, cmd, cycles_per_s=400):
    """(|mean heading-frame velocity - command| per axis over the last second [3, n], base height change, max |roll|, |pitch|)."""
    last = rec["vel"][-cycles_per_s:]
    err = np.abs(last.mean(axis=0) - cmd)
    dz = np.abs(rec["z"] - rec["z"][0]).max(axis=0)
    tilt = np.abs(rec["rpy"][:, 0:2]).max(axis=(0, 1))
    return err, dz, tilt


def test_closed_loop_walks_on_the_cpu(emu, gemu):
    """8 robots, 2 s: forward, backward, lateral, turning and mixed commands.  No failed solve, no negative normal force; over the last
    second the mean base velocity is within 0.05 m/s of the command and the mean yaw rate within 0.1 rad/s; the base height stays
    within 5 cm of the start; |roll|, |pitch| < 0.15 rad."""
    cemu = ContactEmu()
    rec = walk_on_cpu(emu, cemu, gemu, COMMANDS, 800)
    err, dz, tilt = tracking(rec, COMMANDS)
    print("CPU walk: velocity errors x %s, y %s, yaw %s; max |dz| %.3f m, max tilt %.3f rad, min fz %.2f N, max pen %.2f mm"
          % (np.round(err[0], 3), np.round(err[1], 3), np.round(err[2], 3), dz.max(), tilt.max(), rec["fzmin"].min(), 1e3 * rec["pen"].max()))
    assert rec["fzmin"].min() >= 0.0
    assert (err[0:2] <= 0.05).all() and (err[2] <= 0.1).all(), err
    assert (dz < 0.05).all() and (tilt < 0.15).all(), (dz, tilt)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("ground", ["flat", "slope"])
def test_gpu_matches_emulation_host_and_device_pointers(gpu_batch, gemu, ground):
    """4096 robots x 100 cycles of wandering states, random commands, start offsets and contact flags: the kernels through the C ABI
    (host pointers, and device pointers) against the host build of the same source.  Integers equal, doubles to 1e-12 relative."""
    import torch
    from wbc_quadruped_dob_b200 import api
    n, cycles = 4096, 100
    dev = torch.device("cuda", 0)
    T = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    rng = np.random.default_rng(71)
    G = dict(DEFAULTS, stance_cycles=20, swing_cycles=16)
    gp = api.GaitParams(**G)
    drift = Drift(n, 72)
    st = drift.st
    terrain = plane_d = None
    if ground == "slope":
        terrain, plane_d = _slope(n, 73, GR.kinematics(st)[2], 10.0)
    k0 = rng.integers(0, 72, n).astype(np.int32)
    ref, rstatus = gemu.init(G, st, k0, terrain, plane_d)
    hgs = gpu_batch.gait_state(n)
    dgs = gpu_batch.gait_state(n, device=dev)
    hstatus, dstatus = np.full(n, 7, np.int32), torch.full((n,), 7, dtype=torch.int32, device=dev)
    gpu_batch.gait_init({k: st[k] for k in STATE}, hgs, k0, terrain, plane_d, params=gp, status=hstatus)
    gpu_batch.gait_init({k: T(st[k]) for k in STATE}, dgs, T(k0), T(terrain), T(plane_d), params=gp, status=dstatus)
    assert gpu_batch.last_launches() == 1 and (rstatus == 0).all()
    for got, s in ((hgs, hstatus), ({k: v.cpu().numpy() for k, v in dgs.items()}, dstatus.cpu().numpy())):
        assert (s == 0).all()
        _assert_same(got, ref, "init %s" % ground)
    dout = {"mode": torch.zeros(n, dtype=torch.int32, device=dev), **{k: torch.zeros(6, n, dtype=torch.float64, device=dev) for k in GR.OUT}}
    for c in range(cycles):
        cmd = np.vstack([rng.uniform(-0.4, 0.4, n), rng.uniform(-0.2, 0.2, n), rng.uniform(-0.6, 0.6, n)])
        contact = ((rng.uniform(size=(4, n)) < 0.4) * rng.integers(1, 3, (4, n))).astype(np.int32)
        st = drift.next()
        rout, rstatus = gemu.step(G, ref, st, cmd, contact, terrain, plane_d)
        hout = gpu_batch.gait_step({k: st[k] for k in STATE}, hgs, cmd, contact, terrain, plane_d, params=gp, status=hstatus)
        gpu_batch.gait_step({k: T(st[k]) for k in STATE}, dgs, T(cmd), T(contact), T(terrain), T(plane_d), out=dout, params=gp, status=dstatus)
        for what, gs_, out_, s in (("host", hgs, hout, hstatus),
                                   ("device", {k: v.cpu().numpy() for k, v in dgs.items()}, {k: v.cpu().numpy() for k, v in dout.items()},
                                    dstatus.cpu().numpy())):
            assert (s == 0).all() and (rstatus == 0).all()
            _assert_same(gs_, ref, "%s state, cycle %d" % (what, c))
            _assert_same(out_, rout, "%s outputs, cycle %d" % (what, c))


def _torch_feet(base_pos, base_rot, q):
    """Foot points [4, 3, n] (stacked order) of device states: scenarios.forward_kinematics's chain in torch."""
    import torch
    n = q.shape[1]
    R0 = base_rot.T.reshape(n, 3, 3)
    p0 = base_pos.T

    def rot(axis, th):
        a = torch.tensor(axis, dtype=torch.float64, device=q.device)
        K = torch.tensor([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]], dtype=torch.float64, device=q.device)
        s, c = torch.sin(th)[:, None, None], torch.cos(th)[:, None, None]
        return torch.eye(3, dtype=torch.float64, device=q.device)[None] + s * K[None] + (1 - c) * (K @ K)[None]
    feet = [None] * 4
    for leg in range(4):
        R1 = R0 @ rot(S._ROLL_AXIS[leg].tolist(), q[leg])
        p1 = p0 + R0 @ torch.tensor(S._HIP_XYZ[leg], dtype=torch.float64, device=q.device)
        R2 = R1 @ rot(S._PITCH_AXIS[leg].tolist(), q[4 + 2 * leg])
        p2 = p1 + R1 @ torch.tensor(S._PITCH_XYZ[leg], dtype=torch.float64, device=q.device)
        R3 = R2 @ rot(S._KNEE_AXIS[leg].tolist(), q[5 + 2 * leg])
        p3 = p2 + R2 @ torch.tensor(S._KNEE_XYZ, dtype=torch.float64, device=q.device)
        feet[GR.FOOT_LEG.index(leg)] = (p3 + R3 @ torch.tensor(S._FOOT_XYZ, dtype=torch.float64, device=q.device)).T
    return torch.stack(feet)


def walking_herd(gpu_batch, slope, n=4096, cycles=800, seed=81):
    """4096 robots with commands on a 16 x 16 x 16 grid (vx in [-0.1, 0.1] m/s, vy in [-0.05, 0.05] m/s, omega in [-0.2, 0.2] rad/s:
    the envelope in which >= 99 % of touchdowns land within 2 cm of their targets, DESIGN.md 4.8), random start offsets, a 5-25 N push
    on a quarter of them for 0.2 s, `cycles` cycles of gait_step -> cycle_device -> plant_contact_step, all enqueued with sync=False on
    one stream.  The metrics are accumulated on the device and read once at the end.  A robot-swing counts from its lift-off in the
    run (a robot started inside a swing phase has its feet on the ground); the base height is measured above the ground under it."""
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(seed)
    sc, feet = _standing(n, seed)
    g = np.arange(n)
    cmd = np.vstack([np.linspace(-0.1, 0.1, 16)[g % 16], np.linspace(-0.05, 0.05, 16)[(g // 16) % 16], np.linspace(-0.2, 0.2, 16)[(g // 256) % 16]])
    terrain = plane_d = None
    if slope:
        terrain, plane_d = _slope(n, seed + 1, feet, 10.0)
        sc["terrain"] = terrain
    else:
        sc["base_pos"] = sc["base_pos"] - np.array([[0.0], [0.0], [1.0]]) * feet[:, :, 2].min(axis=1)[None]
    push = np.zeros((6, n))
    pushed = g % 4 == 0
    ang = rng.uniform(0, 2 * np.pi, n)
    mag = rng.uniform(5.0, 25.0, n)
    push[0], push[1] = np.where(pushed, mag * np.cos(ang), 0.0), np.where(pushed, mag * np.sin(ang), 0.0)
    k0 = rng.integers(0, 184, n).astype(np.int32)
    T = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    din = {k: T(v) for k, v in sc.items() if isinstance(v, np.ndarray)}
    din["mode"] = torch.zeros(n, dtype=torch.int32, device=dev)
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    dcmd, dpush, dterrain, dplane = T(cmd), T(push), T(terrain), T(plane_d)
    zero = torch.zeros_like(dpush)
    contact = torch.zeros(4, n, dtype=torch.int32, device=dev)
    diag = torch.zeros(4, n, dtype=torch.float64, device=dev)
    cstatus = torch.zeros(n, dtype=torch.int32, device=dev)
    gstatus = torch.zeros(n, dtype=torch.int32, device=dev)
    gs = gpu_batch.gait_state(n, device=dev)
    P = api_params()
    gpu_batch.set_params(P)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    gpu_batch.gait_init(din, gs, T(k0), dterrain, dplane)
    def height():
        z = din["base_pos"][2]
        if not slope:
            return z
        x, y = din["base_pos"][0], din["base_pos"][1]
        return z - sum((dplane[f] - dterrain[10 * f] * x - dterrain[10 * f + 1] * y) / dterrain[10 * f + 2] for f in range(4)) / 4.0
    z0 = height().clone()
    lifted = torch.zeros(n, dtype=torch.bool, device=dev)
    f64 = dict(dtype=torch.float64, device=dev)
    M = {"fails": torch.zeros(n, dtype=torch.int64, device=dev), "fzmin": torch.full((), 1e300, **f64), "pen": torch.zeros((), **f64),
         "vsum": torch.zeros(3, n, **f64), "dz": torch.zeros(n, **f64), "tilt": torch.zeros(n, **f64), "swings": torch.zeros((), **f64),
         "td": torch.zeros((), **f64), "td_near": torch.zeros((), **f64), "td_count": torch.zeros((), **f64)}
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))          # the tensors above were filled on the default stream
    with torch.cuda.stream(stream):
        h = stream.cuda_stream
        for c in range(cycles):
            prev_phase, prev_landed, prev_tick = gs["phase"][0].clone(), gs["landed"][0].clone(), gs["tick"][0].clone()
            gpu_batch.gait_step(din, gs, dcmd, contact, dterrain, dplane, out=din, status=gstatus, stream=h, sync=False)
            swing = (prev_phase % 2) == 1
            touch = swing & (prev_landed == 0) & (din["mode"] == 0)
            lifted |= swing & (prev_tick == 0)
            ended = swing & lifted & (gs["phase"][0] != prev_phase)
            M["swings"] += ended.sum(); M["td"] += (ended & (din["mode"] == 0)).sum()
            lifted &= ~ended
            ft = _torch_feet(din["base_pos"], din["base_rot"], din["q"])          # the feet the gait saw touch down
            first = torch.where(prev_phase < 2, 0, 1)
            idx = torch.arange(n, device=dev)
            d0 = (ft[first, :, idx] - gs["target"][0:3].T).norm(dim=1)
            d1 = (ft[first + 2, :, idx] - gs["target"][3:6].T).norm(dim=1)
            M["td_count"] += touch.sum(); M["td_near"] += (touch & (d0 < 0.02) & (d1 < 0.02)).sum()
            gpu_batch.cycle_device(din, dout, n, n, stream=h, sync=False)
            push_now = dpush if 300 <= c < 380 else zero
            if slope:
                gpu_batch.plant_contact_step(din, dout["tau"], push_now, terrain=dterrain, plane_d=dplane, n=n, ld=n, substeps=5, contact=contact,
                                             diag=diag, status=cstatus, stream=h, sync=False)
            else:
                gpu_batch.plant_contact_step(din, dout["tau"], push_now, n=n, ld=n, substeps=5, contact=contact, diag=diag, status=cstatus,
                                             stream=h, sync=False)
            M["fails"] += (dout["status"] != 0).long() + (cstatus != 0).long() + (gstatus != 0).long()
            M["fzmin"] = torch.minimum(M["fzmin"], diag[1].min()); M["pen"] = torch.maximum(M["pen"], diag[0].max())
            if c >= cycles - 400:
                yaw = din["base_rpy"][2]
                v = din["base_vel"]
                M["vsum"] += torch.stack([torch.cos(yaw) * v[0] + torch.sin(yaw) * v[1], -torch.sin(yaw) * v[0] + torch.cos(yaw) * v[1], v[5]])
            M["dz"] = torch.maximum(M["dz"], (height() - z0).abs())
            M["tilt"] = torch.maximum(M["tilt"], din["base_rpy"][0:2].abs().max(dim=0).values)
    stream.synchronize()
    R = {k: v.cpu().numpy() for k, v in M.items()}
    err = np.abs(R["vsum"] / 400 - cmd)
    ok = (err[0] <= 0.05) & (err[1] <= 0.05) & (err[2] <= 0.1) & (R["dz"] < 0.05) & (R["tilt"] < 0.15)
    return R, err, ok


def api_params():
    from wbc_quadruped_dob_b200 import api
    P = api.default_params()
    P.observer_enabled = 0
    P.dcom = DCOM
    return P


def _check_herd(gpu_batch, slope):
    from wbc_quadruped_dob_b200 import api
    try:
        R, err, ok = walking_herd(gpu_batch, slope)
    finally:
        gpu_batch.set_params(api.default_params())
    print("walking herd (%s): failed solves %d, min normal force %.3f N, max penetration %.3f mm, %d / %d robots track (worst |dv| x %.3f "
          "y %.3f m/s, yaw %.3f rad/s, dz %.1f mm, tilt %.3f rad), %d / %d swings end by touchdown, %d / %d touchdowns within 2 cm of target"
          % ("slope" if slope else "flat", R["fails"].sum(), R["fzmin"], 1e3 * R["pen"], ok.sum(), ok.size, err[0].max(), err[1].max(),
             err[2].max(), 1e3 * R["dz"].max(), R["tilt"].max(), R["td"], R["swings"], R["td_near"], R["td_count"]))
    assert R["fails"].sum() == 0
    assert R["fzmin"] >= 0.0 and R["pen"] < 2e-3
    assert ok.mean() >= 0.99
    assert R["td"] >= 0.99 * R["swings"]
    assert R["td_near"] >= 0.99 * R["td_count"]


@pytest.mark.gpu
def test_walking_herd_on_flat_ground(gpu_batch):
    _check_herd(gpu_batch, slope=False)


@pytest.mark.gpu
def test_walking_herd_on_a_slope_per_robot(gpu_batch):
    """The same herd, each robot on its own slope of up to 10 deg: one terrain array for the gait, the controller and the plant."""
    _check_herd(gpu_batch, slope=True)


class _FakeDevice:
    """Stands in for a CUDA tensor in the side check (which looks only at is_cuda): never dereferenced."""
    is_cuda = True
    shape = (12, 4)

    def data_ptr(self):
        return 0


def test_gait_wrapper_refuses_arrays_from_the_other_side():
    """gait_init / gait_step take the host or the device path from state["q"]; an array of the other side would reach the kernel as a
    pointer of this side, so the wrapper refuses the mix before any call (checked without a ctx: the check is the struct builder's)."""
    from wbc_quadruped_dob_b200 import api
    n = 4
    st = _steady(n)
    hgs = api.WbcBatch.gait_state(n)
    api.WbcBatch._gait_structs(st, hgs, {"cmd": np.zeros((3, n)), "contact": None})
    with pytest.raises(api.WbcError, match="'cmd' is device memory"):
        api.WbcBatch._gait_structs(st, hgs, {"cmd": _FakeDevice()})
    dst = {k: _FakeDevice() for k in STATE}
    dgs = {k: _FakeDevice() for k in hgs}
    api.WbcBatch._gait_structs(dst, dgs, {"cmd": _FakeDevice()})
    for name in ("cmd", "contact", "terrain", "k0", "status", "mode"):
        with pytest.raises(api.WbcError, match="'%s' is host memory" % name):
            api.WbcBatch._gait_structs(dst, dgs, {name: np.zeros((3, n))})
    with pytest.raises(api.WbcError, match="'phase' is host memory"):
        api.WbcBatch._gait_structs(dst, {**dgs, "phase": np.zeros((1, n), np.int32)}, {})


BAD_GAIT_PARAMS = [("stance_cycles", 0), ("stance_cycles", -1), ("stance_cycles", (1 << 20) + 1), ("swing_cycles", 1), ("swing_cycles", 0),
                   ("swing_cycles", (1 << 20) + 1), ("leash", 0.0), ("leash", -0.01)] + \
                  [(k, v) for k in ("step_height", "k_v", "max_step", "acc_lin", "acc_yaw", "leash") for v in (np.nan, np.inf, -np.inf)] + \
                  [(k, -1e-6) for k in ("step_height", "k_v", "max_step", "acc_lin", "acc_yaw")]
EDGE_GAIT_PARAMS = dict(stance_cycles=1, swing_cycles=2, step_height=0.0, k_v=0.0, max_step=0.0, acc_lin=0.0, acc_yaw=0.0, leash=1e-300)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["host", "device"])
def test_gpu_invalid_params_return_einval_with_nothing_done(gpu_batch, path):
    """Each invalid parameter in turn (non-finite doubles, stance_cycles < 1, swing_cycles < 2, either above 2^20, a negative step_height,
    k_v, max_step, acc_lin or acc_yaw, leash <= 0) makes gait_init and gait_step raise WbcError (WBC_EINVAL) and leaves the gait state,
    status, mode and the six outputs bit-identical.  The edge of every bound (stance 1, swing 2, zeros, the smallest positive leash) is
    accepted."""
    import torch
    from wbc_quadruped_dob_b200 import api
    n = 64
    dev = torch.device("cuda", 0)
    st = _steady(n, 91)
    _, _, feet = GR.kinematics(st)
    terrain, plane_d = _slope(n, 92, feet, 10.0)
    k0 = np.arange(n, dtype=np.int32)
    cmd = np.vstack([np.full(n, 0.1), np.zeros(n), np.full(n, 0.2)])
    contact = np.ones((4, n), np.int32)
    if path == "device":
        T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        st, terrain, plane_d, k0, cmd, contact = {k: T(v) for k, v in st.items()}, T(terrain), T(plane_d), T(k0), T(cmd), T(contact)
        gs = gpu_batch.gait_state(n, device=dev)
        status = torch.full((n,), 7, dtype=torch.int32, device=dev)
        snap = lambda d: {k: v.cpu().numpy().copy() for k, v in d.items()}
    else:
        gs = gpu_batch.gait_state(n)
        status = np.full(n, 7, np.int32)
        snap = lambda d: {k: np.array(v, copy=True) for k, v in d.items()}
    gpu_batch.gait_init(st, gs, k0, terrain, plane_d, status=status)
    out = gpu_batch.gait_step(st, gs, cmd, contact, terrain, plane_d, status=status)      # real values in every output
    for k in out:
        out[k] += 3 if k == "mode" else 0.25           # ... and values the next call would not write
    before = (snap(gs), snap(out), snap({"status": status}))
    for field, value in BAD_GAIT_PARAMS:
        gp = api.default_gait_params()
        setattr(gp, field, value)
        for call in (lambda: gpu_batch.gait_init(st, gs, k0, terrain, plane_d, params=gp, status=status),
                     lambda: gpu_batch.gait_step(st, gs, cmd, contact, terrain, plane_d, out=out, params=gp, status=status)):
            with pytest.raises(api.WbcError, match=r"failed \(-1\)"):
                call()
            after = (snap(gs), snap(out), snap({"status": status}))
            for b, a in zip(before, after):
                for k in b:
                    assert np.array_equal(b[k], a[k], equal_nan=True), (field, value, k)
    gp = api.GaitParams(**EDGE_GAIT_PARAMS)
    gpu_batch.gait_init(st, gs, k0, terrain, plane_d, params=gp, status=status)
    gpu_batch.gait_step(st, gs, cmd, contact, terrain, plane_d, out=out, params=gp, status=status)
    assert (snap({"s": status})["s"] == 0).all()
