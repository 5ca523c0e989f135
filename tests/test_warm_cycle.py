"""wbc_cycle with WBC_QP_EXACT | WBC_QP_WARM: each instance starts from the active set its index's previous exact-mode cycle left
in the ctx, when that set was solved in the same contact mode.  The result is the same unique optimum as a cold exact cycle (to
the solver's precision), with far fewer additions in the GI loop on a moving state."""
import ctypes as C

import numpy as np
import pytest

from tests import qp_exact as E
from tests.test_qp_exact import assemble
from wbc_quadruped_dob_b200 import api
from wbc_quadruped_dob_b200 import scenarios as S

pytestmark = pytest.mark.gpu
TOL = 1e-9


def gi_adds(info):
    """inequality rows the GI loop added (qp_info [8, n]): all additions less the warm ones and the equalities"""
    return info[1] - info[6] - (info[4] - info[3])


def rel_x(a, b):
    return (np.abs(a - b).max(axis=0) / np.maximum(1.0, np.abs(b).max(axis=0))).max()


def test_rollout_warm_beside_cold(oracle):
    """4 096 robots x 40 cycles of trot_rollout: a warm ctx and a cold-exact ctx on the same inputs."""
    n, steps = 4096, 40
    a = api.WbcBatch(max_batch=n, device=0)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        zero = np.zeros((6, n))
        a.set_observer_state(zero, zero)
        b.set_observer_state(zero, zero)
        prev_mode = None
        gi_w, gi_c, started = [], [], []
        for k in range(steps):
            sc = S.trot_rollout(n, k)
            w = a.cycle(sc, exact=True, warm=True, want=("x", "status", "qp_info"))
            c = b.cycle(sc, exact=True, want=("x", "status", "qp_info"))
            assert (w["status"] == 0).all() and (c["status"] == 0).all()
            d = rel_x(w["x"], c["x"])
            assert d <= TOL, (k, d)
            flag = (w["qp_info"][5] & api.FL_WARM_STARTED) != 0
            assert not flag.any() if k == 0 else flag.any()
            if prev_mode is not None:
                assert not flag[sc["mode"] != prev_mode].any()
                assert flag[sc["mode"] == prev_mode].all()
                gi_w.append(gi_adds(w["qp_info"]).mean())
                gi_c.append(gi_adds(c["qp_info"]).mean())
                started.append(flag.mean())
            assert (c["qp_info"][6] == 0).all() and (c["qp_info"][7] == 0).all()
            prev_mode = sc["mode"].copy()
            if k == steps - 1:
                idx = np.arange(0, n, 32)
                sco = dict(sc, obs_yd=np.zeros((6, n)), obs_yw=np.zeros((6, n)))   # the assembly takes w itself
                qps = assemble(oracle, sco, idx, w=[w["w"][:, i] for i in idx])
                e = max(E.err(w["x"][:, i], E.exact_qp(Q, cc, L, neq, x0=w["x"][:, i])[0]) for i, (Q, cc, L, neq) in zip(idx, qps))
                assert e <= TOL, e
        print("rollout 4096 x %d: warm-started %.4f of instances; mean GI additions warm %.2f, cold %.2f"
              % (steps, np.mean(started), np.mean(gi_w), np.mean(gi_c)))
        assert np.mean(gi_w) < 0.5 * np.mean(gi_c)
    finally:
        a.close()
        b.close()


def test_checkpoint_restores_the_next_warm_cycle():
    n = 2048
    a = api.WbcBatch(max_batch=n, device=0)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        zero = np.zeros((6, n))
        a.set_observer_state(zero, zero)
        for k in range(3):
            a.cycle(S.trot_rollout(n, k), exact=True, warm=True)
        sets = a.get_active_set(n)
        assert (sets[3] > 0).all() and sets[:3].any()
        yd, yw = a.get_observer_state(n)
        b.set_observer_state(yd, yw)
        b.set_active_set(sets)
        assert np.array_equal(b.get_active_set(n), sets)
        sc = S.trot_rollout(n, 3)
        ra = a.cycle(sc, exact=True, warm=True)
        rb = b.cycle(sc, exact=True, warm=True)
        for key in ra:
            assert np.array_equal(ra[key], rb[key]), key
        assert np.array_equal(a.get_active_set(n), b.get_active_set(n))
    finally:
        a.close()
        b.close()


def test_dispatch_state_default_warm_default():
    """default -> warm -> default on one ctx: the last cycle is bit-identical to a fresh ctx's default cycle."""
    n = 6000
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=23)
    a = api.WbcBatch(max_batch=n, device=0)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        for exact in (False, True):
            a.set_observer_state(sc["obs_yd"], sc["obs_yw"])
            a.cycle(sc, exact=exact, warm=exact)
        yd, yw = a.get_observer_state(n)
        sets = a.get_active_set(n)
        last = a.cycle(sc)
        assert np.array_equal(a.get_active_set(n), sets)          # default cycles leave the stored sets alone
        b.set_observer_state(yd, yw)
        fresh = b.cycle(sc)
        for k in fresh:
            assert np.array_equal(last[k], fresh[k]), k
    finally:
        a.close()
        b.close()


def _raw_cycle(batch, sc, flags):
    """wbc_cycle through the C ABI with the given flags (host pointers); returns (rc, outputs)"""
    n = int(sc["mode"].shape[0])
    keep = []
    ins = batch._inputs_struct(sc, n, keep)
    out = {"tau": np.full((12, n), 7.25), "w": np.full((6, n), 7.25), "x": np.full((30, n), 7.25), "status": np.full(n, 5, np.int32)}
    o = api._Outputs()
    for k in ("tau", "w", "x", "qp_obj", "status", "qp_info", "qp_flops", "w3"):
        setattr(o, k, api._ptr(out.get(k)))
    o.ld = n
    rc = batch.lib.wbc_cycle(batch.h, n, C.byref(ins), C.byref(o), None, flags)
    return rc, out


def test_warm_without_exact_is_refused_with_no_side_effects(gpu_batch):
    n = 512
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), seed=26)
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    gpu_batch.cycle(sc, exact=True)
    sets = gpu_batch.get_active_set(n)
    yd, yw = gpu_batch.get_observer_state(n)
    for flags in (api.QP_WARM, api.QP_WARM | api.FIFO_DISPATCH):
        rc, out = _raw_cycle(gpu_batch, sc, flags)
        assert rc == -1
        assert (out["tau"] == 7.25).all() and (out["w"] == 7.25).all() and (out["x"] == 7.25).all() and (out["status"] == 5).all()
    assert np.array_equal(gpu_batch.get_active_set(n), sets)
    for s0, s1 in zip((yd, yw), gpu_batch.get_observer_state(n)):
        assert np.array_equal(s0, s1)
    with pytest.raises(api.WbcError):
        gpu_batch.cycle(sc, warm=True)


def test_failures_and_hold_tau(gpu_batch):
    n = 64
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), seed=24)
    bad = dict(sc)
    bad["mode"] = sc["mode"].copy(); bad["mode"][3] = 7
    bad["q"] = sc["q"].copy(); bad["q"][2, 5] = np.nan
    res = {}
    for warm in (False, True):
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        gpu_batch.cycle(sc, exact=True)                          # every instance has a stored set
        assert (gpu_batch.get_active_set(n)[3] > 0).all()
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        res[warm] = gpu_batch.cycle(bad, exact=True, warm=warm)
        sets = gpu_batch.get_active_set(n)
        assert not sets[:, [3, 5]].any()                          # a refused instance stores "none"
        assert (np.delete(sets[3], [3, 5]) > 0).all()
    # refused instances as in cold exact mode; the others are the same optimum (to the solver's precision, not bit for bit)
    for k in ("w", "status"):
        assert np.array_equal(res[True][k], res[False][k], equal_nan=True), k
    assert np.array_equal(res[True]["tau"][:, [3, 5]], res[False]["tau"][:, [3, 5]], equal_nan=True)
    assert rel_x(res[True]["x"], res[False]["x"]) <= TOL
    assert rel_x(np.delete(res[True]["tau"], [3, 5], axis=1), np.delete(res[False]["tau"], [3, 5], axis=1)) <= 1e-8
    assert res[True]["status"][3] == -20 and res[True]["status"][5] == -21
    assert not res[True]["x"][:, [3, 5]].any()
    assert ((res[True]["qp_info"][5] & api.FL_WARM_STARTED) != 0).sum() == n - 2
    p = api.default_params()
    p.hold_tau_on_failure = 1
    gpu_batch.set_params(p)
    try:
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        good = gpu_batch.cycle(sc, exact=True, warm=True)
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        held = gpu_batch.cycle(bad, exact=True, warm=True)
    finally:
        gpu_batch.set_params(api.default_params())
    assert np.array_equal(held["tau"][:, [3, 5]], good["tau"][:, [3, 5]])


def test_device_path_equals_host_path():
    import torch
    n = 1024
    a = api.WbcBatch(max_batch=n, device=0)
    b = api.WbcBatch(max_batch=n, device=0)
    dev = torch.device("cuda", 0)
    try:
        zero = np.zeros((6, n))
        a.set_observer_state(zero, zero)
        b.set_observer_state(zero, zero)
        for k in range(3):
            sc = S.trot_rollout(n, k)
            host = a.cycle(sc, exact=True, warm=True, want=("x", "status", "qp_info"))
            din = {key: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for key, v in sc.items() if isinstance(v, np.ndarray) and key != "mode"}
            din["mode"] = torch.from_numpy(np.ascontiguousarray(sc["mode"], dtype=np.int32)).to(dev)
            dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
                    "x": torch.zeros(30, n, dtype=torch.float64, device=dev), "status": torch.zeros(n, dtype=torch.int32, device=dev),
                    "qp_info": torch.zeros(8, n, dtype=torch.int32, device=dev)}
            b.cycle_device(din, dout, n, n, exact=True, warm=True)
            for key in ("tau", "w", "x", "status", "qp_info"):
                assert np.array_equal(dout[key].cpu().numpy(), host[key]), (k, key)
        assert np.array_equal(a.get_active_set(n), b.get_active_set(n))
    finally:
        a.close()
        b.close()


def test_closed_loop_trot_warm_mode(gpu_batch):
    """test_exact_cycle's 320-cycle closed-loop trot through the forward-dynamics plant, in warm mode; a cold-exact ctx solves
    every visited state and its x agrees to 1e-9."""
    import torch
    from tests.test_fdyn_plant import trot_in_place_targets
    n, P, height = 4096, 40, 0.03
    sched = [S.MODE_STANCE, S.MODE_SWING_BR_FL, S.MODE_STANCE, S.MODE_SWING_BL_FR]
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=False, seed=43)
    sc["dq"] = np.zeros((12, n)); sc["base_vel"] = np.zeros((6, n))
    com, _ = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"] = np.vstack([com.T, sc["base_rpy"]])
    sc["com_des_vel"] = np.zeros((6, n)); sc["com_des_acc"] = np.zeros((6, n))
    sc["foot_force"] = np.zeros((12, n)); sc["foot_force"][2::3] = S.TOTAL_MASS * 9.8 / 4.0
    rng = np.random.default_rng(10)
    push = np.zeros((6, n))
    push[0] = (5.0 + rng.integers(0, 20, n)) * rng.choice([-1.0, 1.0], n)
    push[1] = (5.0 + rng.integers(0, 10, n)) * rng.choice([-1.0, 1.0], n)
    dev = torch.device("cuda", 0)
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}

    def outs():
        return {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
                "x": torch.zeros(30, n, dtype=torch.float64, device=dev), "status": torch.zeros(n, dtype=torch.int32, device=dev),
                "qp_info": torch.zeros(8, n, dtype=torch.int32, device=dev)}
    dout, cout = outs(), outs()
    dpush = torch.from_numpy(push).to(dev)
    zero = torch.zeros_like(dpush)
    diag = torch.zeros(2, n, dtype=torch.float64, device=dev)
    cold = api.WbcBatch(max_batch=n, device=0)
    try:
        gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
        cold.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
        fails, worst, anchor, gi_w, gi_c = 0, 0.0, None, 0, 0
        for c in range(8 * P):
            mode = sched[(c // P) % 4]
            if c % P == 0:
                host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
                _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
                din["mode"] = torch.full((n,), mode, dtype=torch.int32, device=dev)
            sp, sv, sa = trot_in_place_targets(anchor, mode, (c % P) / P, P * 0.0025, height)
            din["sw_des_pos"].copy_(torch.from_numpy(sp)); din["sw_des_vel"].copy_(torch.from_numpy(sv)); din["sw_des_acc"].copy_(torch.from_numpy(sa))
            gpu_batch.cycle_device(din, dout, n, n, exact=True, warm=True)
            cold.cycle_device(din, cout, n, n, exact=True)
            fails += int((dout["status"] != 0).sum().item())
            xw, xc = dout["x"].cpu().numpy(), cout["x"].cpu().numpy()
            worst = max(worst, rel_x(xw, xc))
            iw, ic = dout["qp_info"].cpu().numpy(), cout["qp_info"].cpu().numpy()
            gi_w += int(gi_adds(iw).sum()); gi_c += int(gi_adds(ic).sum())
            gpu_batch.plant_dynamics_step(din, dout["tau"], dpush if P <= c < 3 * P else zero, n=n, ld=n, substeps=5, gamma=100.0, diag=diag)
        print("closed-loop trot, warm mode: %d robots x %d cycles, failed solves %d, worst x distance to cold exact %.3e, "
              "GI additions per solve warm %.2f, cold %.2f" % (n, 8 * P, fails, worst, gi_w / (8 * P * n), gi_c / (8 * P * n)))
        assert fails == 0 and worst <= TOL
        assert gi_w < gi_c
    finally:
        cold.close()
