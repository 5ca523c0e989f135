"""The contact plant (wbc_plant_contact_step, csrc/wbc_contact.cuh): unilateral, frictional point contacts at the feet.

CPU: the kernel's source compiled for the host (tests/host_emu/contact_emu.cpp) against an independent reference
(tests/contact_ref.py: the oracle's dense dynamics and a certified primal active-set QP), and physics checks on the emulation:
free fall, landing, no pull, stick, slip.  GPU: the kernel against the emulation, and the controller closed through the plant in a
trot in place whose swing phases end at touchdown."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import contact_ref as CR
from tests import util
from wbc_quadruped_dob_b200 import scenarios as S

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
STATE = ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")


class _ContactParams(C.Structure):
    _fields_ = [("beta", C.c_double), ("eps", C.c_double), ("margin", C.c_double), ("max_iter", C.c_int)]


class ContactEmu:
    """g++ build of contact_step_instance (test infrastructure only)."""

    def __init__(self):
        so = os.path.join(util.EMU_DIR, "libcontact_emu.so")
        util._build_emu(os.path.join(util.EMU_DIR, "contact_emu.cpp"), so)
        self.lib = C.CDLL(so)
        self.lib.emu_contact_step.argtypes = [C.POINTER(util.EmuParams), C.POINTER(_ContactParams), C.c_int, C.c_long] + [_dp] * 7 + \
            [_dp, _dp, _dp, _dp, _ip, _dp, _ip, C.c_int]
        self.lib.emu_contact_step.restype = None

    def step(self, st, tau, push, ground_z=None, mu=None, nsub=5, params=None, cp=(0.2, 1e-8, 2e-3, 64)):
        """Advances a copy of st; returns (next state incl. foot_force, contact [4, n], diag [4, n], status [n])."""
        n = st["q"].shape[1]
        P = params or util.emu_default_params()
        out = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
        out["foot_force"] = np.array(st.get("foot_force", np.zeros((12, n))), dtype=np.float64, order="C")
        contact, diag, status = np.zeros((4, n), np.int32), np.zeros((4, n)), np.zeros(n, np.int32)
        keep = [np.ascontiguousarray(a, dtype=np.float64) if a is not None else None for a in (tau, push, ground_z, mu)]
        d = lambda a: None if a is None else a.ctypes.data_as(_dp)
        self.lib.emu_contact_step(C.byref(P), C.byref(_ContactParams(*cp)), n, n, *[d(out[k]) for k in STATE], d(out["foot_force"]),
                                  *[d(a) for a in keep], contact.ctypes.data_as(_ip), d(diag), status.ctypes.data_as(_ip), int(nsub))
        return out, contact, diag, status


@pytest.fixture(scope="module")
def cemu():
    return ContactEmu()


def mixed_states(n, seed):
    """Feet above the ground, on it and up to 3 mm below it (a ground plane per foot), mu in [0.05, 1], torques and pushes."""
    rng = np.random.default_rng(seed)
    sc = S.make(n, mode_mix=(0.34, 0.33, 0.33), pushes=False, seed=seed)
    st = {k: np.ascontiguousarray(sc[k]) for k in STATE}
    z = CR.foot_heights(st)
    gap = rng.choice([-0.003, 0.0, 0.001, 0.004], size=(4, n)) * rng.uniform(0.0, 1.0, (4, n))
    gap[rng.uniform(size=(4, n)) < 0.15] = 0.0
    ground_z = z - gap
    mu = rng.uniform(0.05, 1.0, n)
    tau = rng.normal(0.0, 4.0, (12, n))
    push = rng.normal(0.0, 15.0, (6, n))
    return st, tau, push, ground_z, mu


def test_foot_points_are_the_oracles(oracle):
    """forward_kinematics places the very foot points whose gaps the plant measures (the oracle's foot frames)."""
    O = oracle
    st, *_ = mixed_states(6, 3)
    z = CR.foot_heights(st)
    for i in range(6):
        one = {k: st[k][:, i:i + 1] for k in STATE}
        one.update({k: np.zeros((m, 1)) for k, m in CR._ZERO_FIELDS.items()})
        one["mode"] = np.zeros(1, np.int32)
        fp = np.array(O.update_only(one, 0).foot_pos).reshape(4, 3)
        assert np.abs(fp[:, 2] - z[:, i]).max() < 1e-12


def test_emulation_matches_the_independent_reference(cemu, oracle):
    """512 mixed states in groups of one to five substeps: forces, state and contact flags equal the certified reference, and every
    kernel-side contact QP meets its KKT conditions to 1e-10 (scaled)."""
    n = 512
    st, tau, push, gz, mu = mixed_states(n, 11)
    groups = np.array_split(np.arange(n), 5)
    nflags = np.zeros(3, int)
    for nsub, idx in enumerate(groups, start=1):
        sub = {k: np.ascontiguousarray(v[:, idx]) for k, v in st.items()}
        got, flags, diag, status = cemu.step(sub, tau[:, idx], push[:, idx], gz[:, idx], mu[idx], nsub=nsub)
        ref, rflags, _ = CR.contact_step(oracle, sub, tau[:, idx], push[:, idx], gz[:, idx], mu[idx], nsub)
        assert (status == 0).all()
        assert (flags == rflags).all(), np.argwhere(flags != rflags)
        fs = np.abs(ref["foot_force"]).max()
        assert np.abs(got["foot_force"] - ref["foot_force"]).max() <= 1e-9 * max(1.0, fs), nsub
        for k in STATE:
            assert np.abs(got[k] - ref[k]).max() <= 1e-10 * max(1.0, np.abs(ref[k]).max()), (nsub, k, np.abs(got[k] - ref[k]).max())
        assert diag[2].max() <= 1e-10, diag[2].max()
        assert diag[1].min() >= 0.0 and diag[0].max() >= 0.0
        nflags += np.bincount(flags.ravel(), minlength=3)
    assert (nflags > 20).all(), nflags                     # no contact, sticking and sliding feet all occur


def test_warm_start_and_cold_start_give_the_same_optimum(cemu, oracle):
    """Five substeps (warm-started from the previous one's rows) against five calls of one substep each with dt / 5 -- the same
    arithmetic, each solve cold -- cannot be compared bit for bit, so the warm run is held to the certified reference instead,
    and its iteration count must not exceed the cold runs'."""
    n = 64
    st, tau, push, gz, mu = mixed_states(n, 12)
    got, flags, diag, status = cemu.step(st, tau, push, gz, mu, nsub=5)
    ref, rflags, _ = CR.contact_step(oracle, st, tau, push, gz, mu, 5)
    assert (status == 0).all() and (flags == rflags).all()
    assert np.abs(got["q"] - ref["q"]).max() <= 1e-10
    P = util.emu_default_params()
    P.obs_dt = 0.0005
    cold_iters = np.zeros(n)
    cur = st
    for _ in range(5):
        cur, _, d1, s1 = cemu.step(cur, tau, push, gz, mu, nsub=1, params=P)
        assert (s1 == 0).all()
        cold_iters += d1[3]
    assert diag[3].sum() <= cold_iters.sum(), (diag[3].sum(), cold_iters.sum())


def test_failures_leave_the_state_untouched(cemu):
    n = 8
    st, tau, push, gz, mu = mixed_states(n, 13)
    tau[3, 2] = np.nan
    gz[:, 5] = S.forward_kinematics(st["base_pos"], st["base_rot"], st["q"])[1][5, :, 2] + 0.001       # all four feet in contact
    got, flags, diag, status = cemu.step(st, tau, push, gz, mu, nsub=3)
    assert status[2] == -21 and (flags[:, 2] == 0).all()
    for k in STATE:
        assert (got[k][:, 2] == st[k][:, 2]).all()
    got, flags, diag, status = cemu.step(st, tau, push, gz, mu, nsub=3, cp=(0.2, 1e-8, 2e-3, 1))
    assert status[5] == -100
    for k in STATE:
        assert (got[k][:, 5] == st[k][:, 5]).all()


def test_free_fall(cemu, oracle):
    """Every foot above its ground plane by more than the margin: no contact force, flags 0, no dual step, and the step is the
    reference's unconstrained one."""
    n = 16
    st, tau, push, _, mu = mixed_states(n, 14)
    gz = CR.foot_heights(st) - 0.05
    got, flags, diag, status = cemu.step(st, tau, push, gz, mu, nsub=5)
    ref, rflags, _ = CR.contact_step(oracle, st, tau, push, gz, mu, 5)
    assert (status == 0).all() and (flags == 0).all() and (rflags == 0).all()
    assert (got["foot_force"] == 0.0).all() and diag[3].max() == 0.0
    for k in STATE:
        assert np.abs(got[k] - ref[k]).max() <= 1e-10 * max(1.0, np.abs(ref[k]).max()), k


def _standing(n, seed, lift=0.0):
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=seed)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    sc["obs_yd"] = np.zeros((6, n)); sc["obs_yw"] = np.zeros((6, n))
    gz = feet[:, :, 2].T.copy()
    sc["base_pos"] = sc["base_pos"] + np.array([[0.0], [0.0], [lift]])
    return sc, gz


def _closed_loop(emu, cemu, sc, gz, mu, cycles, push=None, nsub=5, each=None, dcom=None):
    """The controller (host emulation of wbc_cycle, observer off) closed through the contact plant; calls each(c, sc, out)."""
    n = sc["q"].shape[1]
    P = util.emu_default_params()
    P.observer_enabled = 0
    if dcom is not None:
        P.dcom = dcom
    push = np.zeros((6, n)) if push is None else push
    for c in range(cycles):
        res = emu.cycle(sc, params=P)
        assert (res["status"] == 0).all()
        before = {k: sc[k].copy() for k in STATE}
        out = cemu.step(sc, res["tau"], push, gz, np.full(n, mu), nsub=nsub)
        assert (out[3] == 0).all()
        for k in STATE + ("foot_force",):
            sc[k] = out[0][k]
        if each:
            each(c, before, out)
    return sc


def test_landing(emu, cemu):
    """A robot held by the standing controller and dropped from 2 cm lands and settles: after 0.5 s it penetrates less than 1 mm,
    its base moves slower than 1 cm/s, and no normal force was ever negative.  The CoM gains are made critically damped
    (dcom = 2 sqrt(kcom m) instead of the reference's 50, a damping ratio of 0.11 whose CoM rings for seconds whatever the plant)."""
    n = 3
    sc, gz = _standing(n, 51, lift=0.02)
    fzmin, pen = [1e9], [0.0]

    def each(c, before, out):
        fzmin[0] = min(fzmin[0], out[2][1].min())
        pen[0] = max(pen[0], out[2][0].max())
    sc = _closed_loop(emu, cemu, sc, gz, 0.6, 200, each=each, dcom=2.0 * np.sqrt(2500.0 * S.TOTAL_MASS))
    final_pen = np.maximum(0.0, gz - CR.foot_heights(sc)).max()
    assert final_pen < 1e-3, final_pen
    assert np.abs(sc["base_vel"][:3]).max() < 0.01, sc["base_vel"][:3]
    assert fzmin[0] >= 0.0
    print("landing: max penetration %.2f mm during, %.3f mm at 0.5 s; base speed %.2e m/s" % (1e3 * pen[0], 1e3 * final_pen, np.abs(sc["base_vel"][:3]).max()))


def test_no_pull(emu, cemu):
    """Torques that lift one leg (J_leg' (0, 0, 40 N) on it, the standing controller's torques on the others): that foot gets a
    normal force of exactly 0, its gap grows, and its flag becomes 0; the ground never pulls."""
    n, foot = 2, 2
    sc, gz = _standing(n, 52)
    P = util.emu_default_params()
    P.observer_enabled = 0
    tau = emu.cycle(sc, params=P)["tau"]
    from oracle import oracle_py as O
    leg_dofs = [S_dof for S_dof in range(12) if _dof_leg(S_dof) == _stacked_leg(foot)]
    for i in range(n):
        one = {k: sc[k][:, i:i + 1] for k in STATE}
        one.update({k: np.zeros((m, 1)) for k, m in CR._ZERO_FIELDS.items()})
        one["mode"] = np.zeros(1, np.int32)
        Jl = np.array(O.update_only(one, 0).Jac_lin).reshape(12, 18)[3 * foot:3 * foot + 3, 6:]
        tau[leg_dofs, i] = (Jl.T @ np.array([0.0, 0.0, 40.0]))[leg_dofs]
    gaps = []
    st = {k: sc[k] for k in STATE}
    for c in range(20):
        st, flags, diag, status = cemu.step(st, tau, np.zeros((6, n)), gz, np.full(n, 0.6), nsub=5)
        assert (status == 0).all() and diag[1].min() >= 0.0
        gaps.append((CR.foot_heights(st) - gz)[foot])
        if c >= 2:
            assert (st["foot_force"][3 * foot:3 * foot + 3] == 0.0).all() and (flags[foot] == 0).all()
    gaps = np.array(gaps)
    assert (np.diff(gaps[2:], axis=0) > 0.0).all() and (gaps[-1] > 1e-3).all(), gaps[:, 0]


def _dof_leg(d):
    return d if d < 4 else (d - 4) // 2     # DoF order: roll BL, BR, FL, FR, then (pitch, knee) pairs of BL, BR, FL, FR


def _stacked_leg(foot):
    return (1, 0, 2, 3)[foot]          # stacked BR, BL, FL, FR -> canonical leg BL, BR, FL, FR


def test_stick(emu, cemu):
    """mu = 0.6, standing under the controller with no push: all four feet stick for 1 s and drift less than 0.1 mm."""
    n = 2
    sc, gz = _standing(n, 53)
    _, feet0 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    seen = []
    sc = _closed_loop(emu, cemu, sc, gz, 0.6, 400, each=lambda c, b, out: seen.append(out[1].copy()))
    assert (np.array(seen) == 1).all()
    _, feet1 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    drift = np.abs(feet1 - feet0).max()
    assert drift < 1e-4, drift
    print("stick: foot drift %.2e m over 1 s" % drift)


def test_slip(emu, cemu, oracle):
    """mu = 0.05, a 40 N lateral push: the feet slide (flag 2); the tangential impulse of a sliding foot lies on the pyramid's
    boundary, friction does no positive work, and the foot's normal velocity after the step stays within the relaxation's bound
    (target + mu (|v_x| + |v_y|): the pyramid's form of 'mu times the slip speed')."""
    n, mu = 2, 0.05
    sc, gz = _standing(n, 54)
    push = np.zeros((6, n)); push[1] = 40.0
    P = util.emu_default_params()
    P.observer_enabled = 0
    slides = 0
    for c in range(40):
        res = emu.cycle(sc, params=P)
        st = {k: sc[k] for k in STATE}
        ref, rflags, lam = CR.contact_step(oracle, st, res["tau"], push, gz, np.full(n, mu), 1)
        got, flags, diag, status = cemu.step(st, res["tau"], push, gz, np.full(n, mu), nsub=1)
        assert (status == 0).all() and (flags == rflags).all()
        for i in range(n):
            one = {k: st[k][:, i:i + 1] for k in STATE}
            one.update({k: np.zeros((m, 1)) for k, m in CR._ZERO_FIELDS.items()})
            one["mode"] = np.zeros(1, np.int32)
            d = oracle.update_only(one, 0)
            J = np.array(d.Jac_lin).reshape(12, 18)
            v = J @ np.concatenate([got["base_vel"][:, i], got["dq"][:, i]])
            phi = np.array(d.foot_pos).reshape(4, 3)[:, 2] - gz[:, i]
            for k in range(4):
                if flags[k, i] != 2:
                    continue
                slides += 1
                lk, vk = lam[3 * k:3 * k + 3, i], v[3 * k:3 * k + 3]
                assert min(abs(abs(lk[0]) - mu * lk[2]), abs(abs(lk[1]) - mu * lk[2])) <= 1e-9 * lk[2]
                assert lk[0] * vk[0] + lk[1] * vk[1] <= 1e-12 * np.abs(lk).max()
                target = -(1.0 if phi[k] >= 0 else 0.2) * phi[k] / 0.0025
                assert vk[2] - target <= mu * (abs(vk[0]) + abs(vk[1])) * (1 + 1e-6) + 1e-9
        for k in STATE + ("foot_force",):
            sc[k] = got[k]
    assert slides > 40, slides
    print("slip: %d sliding foot-steps" % slides)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_matches_emulation_host_and_device_pointers(gpu_batch, cemu):
    import torch
    from wbc_quadruped_dob_b200 import api
    n = 4096
    st, tau, push, gz, mu = mixed_states(n, 21)
    ref, rflags, rdiag, rstatus = cemu.step(st, tau, push, gz, mu, nsub=5)
    assert (rstatus == 0).all()
    h = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
    h["foot_force"] = np.zeros((12, n))
    contact, diag, status = np.zeros((4, n), np.int32), np.zeros((4, n)), np.full(n, 7, np.int32)
    gpu_batch.plant_contact_step(h, tau, push, ground_z=gz, mu=mu, substeps=5, contact=contact, diag=diag, status=status)
    assert gpu_batch.last_launches() == 1
    dev = torch.device("cuda", 0)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d = {k: T(st[k]) for k in STATE}
    d["foot_force"] = torch.zeros(12, n, dtype=torch.float64, device=dev)
    dc, dd, ds = torch.zeros(4, n, dtype=torch.int32, device=dev), torch.zeros(4, n, dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int32, device=dev)
    gpu_batch.plant_contact_step(d, T(tau), T(push), ground_z=T(gz), mu=T(mu), substeps=5, contact=dc, diag=dd, status=ds)
    for got, c, dg, s in ((h, contact, diag, status), ({k: v.cpu().numpy() for k, v in d.items()}, dc.cpu().numpy(), dd.cpu().numpy(), ds.cpu().numpy())):
        assert (s == 0).all() and (c == rflags).all()
        for k in STATE + ("foot_force",):
            assert np.abs(got[k] - ref[k]).max() <= 1e-10 * max(1.0, np.abs(ref[k]).max()), k
        assert dg[2].max() <= 1e-10 and np.abs(dg[0] - rdiag[0]).max() <= 1e-12
    # defaults: ground at z = 0 and params.mu; the mode array may be absent
    h2 = {k: np.array(st[k], dtype=np.float64, order="C") for k in STATE}
    h2["foot_force"] = np.zeros((12, n))
    gpu_batch.plant_contact_step(h2, tau, push, substeps=2, params=api.default_contact_params())
    ref2, *_ = cemu.step(st, tau, push, np.zeros((4, n)), np.full(n, 0.6), nsub=2)
    assert np.abs(h2["q"] - ref2["q"]).max() <= 1e-10


@pytest.mark.gpu
def test_closed_loop_trot_in_place_through_the_contact_plant(gpu_batch):
    """4096 robots trotting in place (test_fdyn_plant.py's schedule: stance, swing{BR,FL}, stance, swing{BL,FR}, 40 cycles per phase,
    3 cm foot lift, pushes in the second and third phase), closed for 320 cycles through the contact plant.  A robot's swing phase
    ends at the phase end or at touchdown -- both swing feet in contact after mid-swing, read from the plant's contact flags --
    whichever comes first.  No solve fails, no normal force is negative, no foot sinks 2 mm into the ground, the swing feet really
    leave it (no contact at mid-swing, apex >= 2 cm on >= 99 % of robot-swings), and the robots stay up."""
    import torch
    from tests.test_fdyn_plant import trot_in_place_targets
    n, P, height = 4096, 40, 0.03
    sched = [S.MODE_STANCE, S.MODE_SWING_BR_FL, S.MODE_STANCE, S.MODE_SWING_BL_FR]
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=43)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    gz = np.ascontiguousarray(feet[:, :, 2].T)
    base0 = sc["base_pos"].copy()
    rng = np.random.default_rng(10)
    push = np.zeros((6, n))
    push[0] = (5.0 + rng.integers(0, 20, n)) * rng.choice([-1.0, 1.0], n)
    push[1] = (5.0 + rng.integers(0, 10, n)) * rng.choice([-1.0, 1.0], n)
    dev = torch.device("cuda", 0)
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    dpush = torch.from_numpy(push).to(dev)
    zero = torch.zeros_like(dpush)
    dgz = torch.from_numpy(gz).to(dev)
    contact = torch.zeros(4, n, dtype=torch.int32, device=dev)
    diag = torch.zeros(4, n, dtype=torch.float64, device=dev)
    cstatus = torch.zeros(n, dtype=torch.int32, device=dev)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    fails, cfails, fzmin, pen, slips, touchdowns, airborne_mid, mid_checks = 0, 0, 1e9, 0.0, 0, 0, 0, 0
    apex_ok, swings, anchor, apex, landed = 0, 0, None, None, None
    for c in range(8 * P):
        mode = sched[(c // P) % 4]
        s = (c % P) / P
        first, second = (1, 3) if mode == S.MODE_SWING_BL_FR else (0, 2)
        if c % P == 0:
            host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
            _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
            landed = np.zeros(n, bool)
            apex = np.zeros(n)
        if mode != S.MODE_STANCE:
            # a robot whose two swing feet are down after mid-swing has touched down: it is in stance for the rest of the phase
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
        pushed = P <= c < 3 * P
        gpu_batch.plant_contact_step(din, dout["tau"], dpush if pushed else zero, ground_z=dgz, n=n, ld=n, substeps=5, contact=contact, diag=diag,
                                     status=cstatus)
        cfails += int((cstatus != 0).sum().item())
        dg = diag.cpu().numpy()
        fzmin = min(fzmin, float(dg[1].min()))
        pen = max(pen, float(dg[0].max()))
        cf = contact.cpu().numpy()
        slips += int((cf == 2).sum())
        if mode != S.MODE_STANCE:
            host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
            _, ft = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
            lift = np.minimum(ft[:, first, 2] - gz[first], ft[:, second, 2] - gz[second])
            apex = np.maximum(apex, lift)
            if c % P == P // 2:
                mid_checks += 2 * n
                airborne_mid += int((cf[first] == 0).sum() + (cf[second] == 0).sum())
            if c % P == P - 1:
                swings += n
                apex_ok += int((apex >= 0.02).sum())
    pos = din["base_pos"].cpu().numpy()
    rpy = din["base_rpy"].cpu().numpy()
    print("closed-loop trot through the contact plant: %d robots x %d cycles, failed solves %d / %d, min normal force %.3f N, max penetration %.3f mm, "
          "swing feet airborne at mid-swing %d / %d, apex >= 2 cm on %d / %d robot-swings, %d sliding foot-cycles, %d touchdowns before the phase end, "
          "max |base drift| %.1f mm, max |rpy - rpy0| %.3f rad"
          % (n, 8 * P, fails, cfails, fzmin, 1e3 * pen, airborne_mid, mid_checks, apex_ok, swings, slips, touchdowns,
             1e3 * np.abs(pos - base0).max(), np.abs(rpy - sc["base_rpy"]).max()))
    assert fails == 0 and cfails == 0
    assert fzmin >= 0.0 and pen < 2e-3
    assert airborne_mid == mid_checks and apex_ok >= 0.99 * swings
    assert np.abs(pos - base0).max() < 0.08 and np.abs(rpy - sc["base_rpy"]).max() < 0.15
