"""SURVEY.md 8f-2: forward dynamics with hard contacts as the closed-loop plant (stands in for Gazebo + force_plugin's ModelPush,
fp.cpp:124-491; PARITY UNPINNED -- the reference for this stage is a physics engine).  CPU: physics identities of the oracle's
dense, literal formulation.  GPU: the kernel's Schur-complement formulation against it, and the controller closed through it."""
import numpy as np
import pytest

from tests import util
from wbc_quadruped_dob_b200 import scenarios as S


def _standing(n, seed=31):
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=seed)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    return sc


def test_contact_constraint_and_free_fall(oracle):
    n = 12
    sc = S.make(n, mode_mix=(0.34, 0.33, 0.33), pushes=False, seed=5)
    tau = np.random.default_rng(1).normal(0.0, 3.0, (12, n))
    push = np.zeros((6, n)); push[0] = 20.0
    nxt, diag = oracle.fdyn_step(sc, tau, push, nsub=1, gamma=0.0)
    assert diag[:, 0].max() < 1e-9                                  # J nu_dot + Jdqd = 0 at the stance feet
    # one substep with gamma = 0 keeps the contact-point velocity to first order: J nu after = J nu before + O(dt^2)
    for i in range(n):
        d0 = oracle.update_only(sc, i)
        one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
        one.update({k: nxt[k][..., i:i + 1] for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")})
        d1 = oracle.update_only(one, 0)
        fv0, fv1 = np.array(d0.foot_vel).reshape(4, 3), np.array(d1.foot_vel).reshape(4, 3)
        mode = int(sc["mode"][i])
        for f in range(4):
            swing = (mode == 1 and f in (0, 2)) or (mode == 2 and f in (1, 3))
            if not swing:
                assert np.abs(fv1[f] - fv0[f]).max() < 2e-3, (i, f, fv0[f], fv1[f])


def test_energy_balance_under_hard_contacts(oracle):
    """Standing robot at rest, constant joint torques, no push: over a short horizon the change of kinetic + potential energy
    equals the work of the joint torques (rigid bilateral contacts with stationary contact points do no work)."""
    n = 6
    sc = _standing(n)
    rng = np.random.default_rng(7)
    tau = rng.normal(0.0, 2.0, (12, n))
    push = np.zeros((6, n))

    def energy(s):
        e = np.zeros(n)
        for i in range(n):
            d = oracle.update_only(s, i)
            M = np.array(d.M).reshape(18, 18)
            nu = np.concatenate([s["base_vel"][:, i], s["dq"][:, i]])
            e[i] = 0.5 * nu @ M @ nu + S.TOTAL_MASS * 9.8 * np.array(d.com)[2]
        return e
    cur = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    P = oracle.default_params()
    e0 = energy(cur)
    work = np.zeros(n)
    for step in range(8):
        q_before = cur["q"].copy()
        nxt, diag = oracle.fdyn_step(cur, tau, push, params=P, nsub=25, gamma=0.0)
        work += np.einsum("kn,kn->n", tau, nxt["q"] - q_before)
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq"):
            cur[k] = nxt[k]
    e1 = energy(cur)
    assert np.abs((e1 - e0) - work).max() < 2e-2 * max(1e-3, np.abs(work).max()) + 1e-5, (e1 - e0, work)


def test_standing_torques_hold_the_robot_still(oracle, oracle_qp):
    """The controller's own torques through the plant: a robot at rest on four feet, desired CoM = actual CoM, stays at rest."""
    n = 8
    sc = _standing(n)
    com, _ = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["obs_yd"] = np.zeros((6, n)); sc["obs_yw"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    P = oracle.default_params(observer_enabled=0)
    cur = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    for it in range(40):
        res, _ = oracle.run_cycle_batch(cur, P, nthreads=8, solver=oracle_qp)
        nxt, diag = oracle.fdyn_step(cur, res["tau"].T, np.zeros((6, n)), params=P, nsub=5, gamma=100.0)
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force"):
            cur[k] = nxt[k]
        assert diag[:, 1].min() > 0.0                               # every foot keeps pushing on the ground
    assert np.abs(cur["base_pos"] - sc["base_pos"]).max() < 5e-3
    assert np.abs(cur["base_vel"]).max() < 0.1


def test_device_plant_step_matches_oracle_on_the_host(emu, oracle):
    """fdyn_step_instance (the kernel's Schur-complement formulation, compiled for the host) against the oracle's dense
    elimination: one control period of five substeps, all contact modes, torques and pushes."""
    n = 48
    sc = S.make(n, mode_mix=(0.34, 0.33, 0.33), pushes=False, seed=17)
    rng = np.random.default_rng(3)
    tau = rng.normal(0.0, 4.0, (12, n))
    push = rng.normal(0.0, 15.0, (6, n))
    ref, rdiag = oracle.fdyn_step(sc, tau, push, nsub=5, gamma=100.0)
    got, gdiag = emu.fdyn_step(sc, tau, push, nsub=5, gamma=100.0)
    for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq"):
        assert np.abs(got[k] - ref[k]).max() <= 1e-9 * max(1.0, np.abs(ref[k]).max()), k
    assert np.abs(got["foot_force"] - ref["foot_force"]).max() <= 1e-8 * max(1.0, np.abs(ref["foot_force"]).max())
    assert gdiag[0].max() < 1e-8 and np.abs(gdiag[1] - rdiag[:, 1]).max() < 1e-7


@pytest.mark.gpu
def test_gpu_plant_step_matches_oracle(gpu_batch, oracle):
    n = 200
    sc = S.make(n, mode_mix=(0.34, 0.33, 0.33), pushes=False, seed=18)
    rng = np.random.default_rng(4)
    tau = rng.normal(0.0, 4.0, (12, n))
    push = rng.normal(0.0, 15.0, (6, n))
    ref, rdiag = oracle.fdyn_step(sc, tau, push, nsub=5, gamma=100.0)
    st = {k: np.array(sc[k], dtype=np.float64, order="C") for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
    st["foot_force"] = np.zeros((12, n)); st["mode"] = np.ascontiguousarray(sc["mode"], dtype=np.int32)
    diag = np.zeros((2, n))
    gpu_batch.plant_dynamics_step(st, tau, push, substeps=5, gamma=100.0, diag=diag)
    assert gpu_batch.last_launches() == 1
    for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq"):
        assert np.abs(st[k] - ref[k]).max() <= 1e-9 * max(1.0, np.abs(ref[k]).max()), k
    assert np.abs(st["foot_force"] - ref["foot_force"]).max() <= 1e-8 * max(1.0, np.abs(ref["foot_force"]).max())
    assert diag[0].max() < 1e-8


@pytest.mark.gpu
def test_closed_loop_standing_under_pushes_through_the_dynamics_plant(gpu_batch):
    """4096 standing robots, controller (wbc_cycle) closed through the forward-dynamics plant for 400 cycles (1 s), everything
    resident on the GPU: a force_plugin-style horizontal push (fp.cpp:203-310: 5..24 N) acts on every robot for the first 0.3 s.
    The robots stay on their feet (normal forces positive, CoM within a few centimetres, velocities bounded), the observer picks the
    push up while it acts and lets go of it afterwards, and no solve fails."""
    import torch
    n, cycles = 4096, 400
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=41)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, _ = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    rng = np.random.default_rng(9)
    push = np.zeros((6, n))
    push[0] = (5.0 + rng.integers(0, 20, n)) * rng.choice([-1.0, 1.0], n)
    push[1] = (5.0 + rng.integers(0, 10, n)) * rng.choice([-1.0, 1.0], n)
    dev = torch.device("cuda", 0)
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    dpush = torch.from_numpy(push).to(dev)
    zero = torch.zeros_like(dpush)
    diag = torch.zeros(2, n, dtype=torch.float64, device=dev)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    fzmin, w_during = 1e9, None
    for c in range(cycles):
        gpu_batch.cycle_device(din, dout, n, n)
        assert int((dout["status"] != 0).sum().item()) == 0, c
        gpu_batch.plant_dynamics_step(din, dout["tau"], dpush if c < 120 else zero, n=n, ld=n, substeps=5, gamma=100.0, diag=diag)
        fzmin = min(fzmin, float(diag[1].min().item()))
        if c == 119:
            w_during = dout["w"].cpu().numpy()
    w_after = dout["w"].cpu().numpy()
    pos = din["base_pos"].cpu().numpy()
    vel = din["base_vel"].cpu().numpy()
    assert fzmin > 0.0                                                  # no foot ever pulled on the ground
    assert np.abs(pos - sc["base_pos"]).max() < 0.05 and np.abs(vel).max() < 0.5
    # k = 10: after 0.3 s the estimate holds 1 - exp(-3) = 95 % of the horizontal push; 0.7 s after it stopped, (almost) nothing
    rel = np.abs(w_during[:2] - push[:2]).max(axis=0) / np.abs(push[:2]).max(axis=0)
    assert np.median(rel) < 0.25, np.median(rel)
    assert np.abs(w_after[:2]).max() < 0.1 * np.abs(push[:2]).max()
    print("closed loop through the dynamics plant: min normal force %.1f N, max |base drift| %.1f mm, median estimate error while pushed %.1f %%"
          % (fzmin, 1e3 * np.abs(pos - sc["base_pos"]).max(), 100 * np.median(rel)))


def trot_in_place_targets(anchor, mode, s, period_s, height):
    """Swing-foot targets of a trot in place: the two swing feet of `mode` leave their anchor (their position when the phase began,
    [n,4,3] stacked foot order) along height * sin^2(pi s), s in [0,1) the phase fraction.  Returns sw_des_pos/vel/acc [6,n]."""
    n = anchor.shape[0]
    first, second = (1, 3) if mode == S.MODE_SWING_BL_FR else (0, 2)
    pos = np.hstack([anchor[:, first, :], anchor[:, second, :]]).T.copy()
    vel = np.zeros((6, n)); acc = np.zeros((6, n))
    if mode != S.MODE_STANCE:
        w = np.pi / period_s
        pos[2] += height * np.sin(np.pi * s) ** 2; pos[5] += height * np.sin(np.pi * s) ** 2
        vel[2] = vel[5] = height * w * np.sin(2 * np.pi * s)
        acc[2] = acc[5] = 2.0 * height * w * w * np.cos(2 * np.pi * s)
    return pos, vel, acc


@pytest.mark.gpu
def test_closed_loop_trot_under_pushes_through_the_dynamics_plant(gpu_batch, oracle_qp):
    """4096 robots trotting in place (stance, swing{BR,FL}, stance, swing{BL,FR}; 40 cycles per phase, 3 cm foot lift), the
    controller closed through the forward-dynamics plant for 320 cycles with a force_plugin-style horizontal push during the second
    and third phase (fp.cpp:203-310).  Contact modes, active sets and joint states all move.  Every robot stays up and no solve
    fails; on a sub-sample the controller's torques are checked against the oracle on the very states the loop visits."""
    import torch
    from oracle import oracle_py as O
    n, P, height = 4096, 40, 0.03
    sched = [S.MODE_STANCE, S.MODE_SWING_BR_FL, S.MODE_STANCE, S.MODE_SWING_BL_FR]
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=43)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, _ = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    base0 = sc["base_pos"].copy()
    rng = np.random.default_rng(10)
    push = np.zeros((6, n))
    push[0] = (5.0 + rng.integers(0, 20, n)) * rng.choice([-1.0, 1.0], n)
    push[1] = (5.0 + rng.integers(0, 10, n)) * rng.choice([-1.0, 1.0], n)
    dev = torch.device("cuda", 0)
    state_keys = ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force")
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    dpush = torch.from_numpy(push).to(dev)
    zero = torch.zeros_like(dpush)
    diag = torch.zeros(2, n, dtype=torch.float64, device=dev)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    fails, fzmin, worst_tau, checked, anchor, pulls = 0, 1e9, 0.0, 0, None, 0
    sub = np.arange(0, n, 64)
    for c in range(8 * P):
        mode = sched[(c // P) % 4]
        if c % P == 0:       # a phase begins: the contact mode of every robot changes, the swing feet start from where they stand
            host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
            _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
            din["mode"] = torch.full((n,), mode, dtype=torch.int32, device=dev)
        sp, sv, sa = trot_in_place_targets(anchor, mode, (c % P) / P, P * 0.0025, height)
        din["sw_des_pos"].copy_(torch.from_numpy(sp)); din["sw_des_vel"].copy_(torch.from_numpy(sv)); din["sw_des_acc"].copy_(torch.from_numpy(sa))
        if c % 20 == 7:
            # teacher-forced check: the oracle on the states the loop is in right now (observer state included)
            yd, yw = gpu_batch.get_observer_state(n)
            one = {k: din[k].cpu().numpy()[..., sub] for k in din if k not in ("mode",)}
            one["mode"] = np.full(sub.size, mode, dtype=np.int32)
            one["obs_yd"], one["obs_yw"] = yd[:, sub], yw[:, sub]
            ref, _ = O.run_cycle_batch(one, nthreads=8, solver=oracle_qp)
        gpu_batch.cycle_device(din, dout, n, n)
        fails += int((dout["status"] != 0).sum().item())
        if c % 20 == 7:
            tau = dout["tau"].cpu().numpy()[:, sub]
            ok = ref["status"] == 0
            worst_tau = max(worst_tau, float((np.abs(tau[:, ok] - ref["tau"].T[:, ok]) / (1.0 + np.abs(ref["tau"].T[:, ok]))).max()))
            checked += int(ok.sum())
        pushed = P <= c < 3 * P
        gpu_batch.plant_dynamics_step(din, dout["tau"], dpush if pushed else zero, n=n, ld=n, substeps=5, gamma=100.0, diag=diag)
        fzmin = min(fzmin, float(diag[1].min().item()))
        pulls += int((diag[1] < 0.0).sum().item())
    pos = din["base_pos"].cpu().numpy()
    rpy = din["base_rpy"].cpu().numpy()
    vel = din["base_vel"].cpu().numpy()
    print("closed-loop trot through the dynamics plant: %d robots x %d cycles, failed solves %d, min normal force %.1f N (%d robot-cycles below zero), max |base drift| %.1f mm, "
          "max |rpy - rpy0| %.3f rad, teacher-forced torque rel err %.2e over %d robot-cycles"
          % (n, 8 * P, fails, fzmin, pulls, 1e3 * np.abs(pos - base0).max(), np.abs(rpy - sc["base_rpy"]).max(), worst_tau, checked))
    assert fails == 0
    # the plant's contacts are bilateral (unilaterality is not enforced): around a phase change the foot that is about to lift is
    # commanded to zero force and the plant may answer with a slightly negative one; it must stay a rare event of a fraction of a newton
    assert fzmin > -1.0 and pulls < 1e-2 * n * 8 * P
    assert np.abs(pos - base0).max() < 0.08 and np.abs(rpy - sc["base_rpy"]).max() < 0.15 and np.abs(vel).max() < 1.0
    assert checked > 900 and worst_tau < 1e-6


def test_oracle_closed_loop_through_the_dynamics_plant_estimates_the_push(oracle, oracle_qp):
    """BASELINE config 5 through the forward-dynamics plant (bench.py --workload push_sweep --plant dynamics), on the oracle: robots
    holding their pose under a constant horizontal push.  The estimate settles on the push in x and y; in z it settles on
    m (g_acc - |gravity|) = +0.21 N, the reference's two gravity constants (9.81 in estimate(), main.cpp:702; 9.8 in the dynamics,
    main.cpp:855 -- quirk E1) showing through a plant that, unlike the momentum integrator, does not share the observer's."""
    sc = S.push_sweep(n=256 * 8 * 2, start=0)
    idx = np.array([256 * 5, 256 * 5 + 1, 256 * 8 + 256 * 5, 256 * 8 + 256 * 5 + 7])          # gain 50; 5 N and 10 N
    sub = {k: (v[..., idx] if isinstance(v, np.ndarray) else v) for k, v in sc.items() if k != "grid"}
    assert (sub["obs_gain"] == 50.0).all()
    com0, _ = S.forward_kinematics(sub["base_pos"], sub["base_rot"], sub["q"])
    sub["com_des_pos"] = np.vstack([com0.T, sub["base_rpy"]])
    push = sub["push"]
    for c in range(160):
        res, _ = oracle.run_cycle_batch_gains(sub, solver=oracle_qp)
        assert (res["status"] == 0).all()
        sub["obs_yd"], sub["obs_yw"] = res["yd"].T.copy(), res["yw"].T.copy()
        nxt, diag = oracle.fdyn_step(sub, res["tau"].T, push, nsub=5, gamma=100.0)
        assert diag[:, 1].min() > 0.0
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force"):
            sub[k] = nxt[k]
    w = res["w"].T
    assert np.abs(w[:2] - push[:2]).max() < 0.05                               # k = 50: e^-20 of the push is left, plus the robot's sway
    assert np.abs(w[2] - S.TOTAL_MASS * (9.81 - 9.8)).max() < 0.02
    assert np.abs(sub["base_pos"] - sc["base_pos"][:, idx]).max() < 0.01
