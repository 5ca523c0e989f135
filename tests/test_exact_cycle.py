"""wbc_cycle with WBC_QP_EXACT (the dual active-set solver of csrc/qp_dual.cuh in wbc_solve_exact_kernel): the cycle's QP
solutions against the certified optimum x* (tests/qp_exact.py), its torques against the live oracle solving with x*, and
everything around the solve (observer, dispatch state, failure handling) against default mode."""
import ctypes as C

import numpy as np
import pytest

from tests import qp_exact as E
from tests import util
from tests.test_qp_exact import assemble
from wbc_quadruped_dob_b200 import scenarios as S

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _exact_cycle(batch, sc):
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    got = batch.cycle(sc, exact=True)
    assert batch.last_launches() == 2
    batch.solver_shape()
    assert batch.last_solver_kernel == "wbc_solve_exact_kernel"
    return got


def _check_x(what, oracle, got, sc, idx):
    assert (got["status"][idx] == 0).all()
    qps = assemble(oracle, sc, idx, w=[got["w"][:, i] for i in idx])
    x = got["x"][:, idx].T
    e = np.array([E.err(xk, E.exact_qp(Q, c, L, neq, x0=xk)[0]) for (Q, c, L, neq), xk in zip(qps, x)])
    print("%s: %d instances, worst err %.3e" % (what, len(idx), e.max()))
    assert e.max() <= TOL
    assert ((got["qp_info"][5][idx] & 256) != 0).all()


def test_exact_cycle_standing_4096(gpu_batch, oracle):
    sc = S.make_config("standing_4096")
    got = _exact_cycle(gpu_batch, sc)
    _check_x("exact cycle standing_4096", oracle, got, sc, np.arange(4096))
    # where DENSE-AUL converges (stance, Appendix F), the two modes give the same torques
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    ref = gpu_batch.cycle(sc)
    st = np.flatnonzero(sc["mode"] == 0)
    e = util.rel_rows(got["tau"].T[st], ref["tau"].T[st])
    print("standing_4096 stance instances: exact vs default worst tau rel diff %.3e" % e.max())
    assert e.max() <= 1e-6


def test_exact_cycle_mixed_terrain_pushes(gpu_batch, oracle):
    sc = S.make(3000, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=12)
    got = _exact_cycle(gpu_batch, sc)
    _check_x("exact cycle mixed terrain pushes", oracle, got, sc, np.arange(3000))


def test_exact_cycle_trot_65536(gpu_batch, oracle):
    sc = S.make_config("trot_65536")
    got = _exact_cycle(gpu_batch, sc)
    _check_x("exact cycle trot_65536 (every 16th)", oracle, got, sc, np.arange(0, 65536, 16))


def test_exact_cycle_matches_live_oracle_solving_exactly(gpu_batch, oracle):
    """The live oracle's control cycle with its QP solved by qp_exact.exact_qp (a ctypes wbc_qp_fn): tau within 1e-6.  The
    reference is warm-started from the host emulation's x (its cold start can meet a singular KKT system on these degenerate
    vertices); what it returns is certified by the KKT conditions independently of that guess."""
    from tests.test_qp_dual import DualEmu
    dual = DualEmu()

    def solve(Q, c, L, nrows, neq, x, nchol, term):
        Qa = np.ctypeslib.as_array(Q, (900,)).reshape(30, 30).copy()
        ca = np.ctypeslib.as_array(c, (30,)).copy()
        La = np.ctypeslib.as_array(L, (nrows * 31,)).reshape(nrows, 31).copy() if nrows else np.zeros((0, 31))
        xs = E.exact_qp(Qa, ca, La, neq, x0=dual.solve(Qa, ca, La, neq)[0])[0]
        for k in range(30):
            x[k] = xs[k]
        if nchol:
            nchol[0] = 1
        if term:
            term[0] = 2
        return 0
    fn = oracle.QP_FN(solve)
    sc = S.make(512, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=21)
    got = _exact_cycle(gpu_batch, sc)
    ref, _ = oracle.run_cycle_batch(sc, nthreads=1, solver=fn)
    e = util.rel_rows(got["tau"].T, ref["tau"])
    print("exact cycle vs live oracle with exact QPs: worst tau rel err %.3e" % e.max())
    assert e.max() <= 1e-6
    assert np.abs(got["w"].T - ref["w"]).max() <= util.TOL_OBS * max(1.0, np.abs(ref["w"]).max())


def test_observer_identical_to_default(gpu_batch):
    sc = S.make(2048, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=22)
    outs, states = [], []
    for exact in (False, True):
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        outs.append(gpu_batch.cycle(sc, exact=exact))
        states.append(gpu_batch.get_observer_state(2048))
    assert np.array_equal(outs[0]["w"], outs[1]["w"])
    for a, b in zip(states[0], states[1]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("n,kernel", [(6000, "wbc_solve_kernel"), (49152, "wbc_solve_staged_kernel")])
def test_dispatch_state_default_exact_default(n, kernel):
    """default -> exact -> default on one ctx: the last cycle is bit-identical to a fresh ctx's default cycle, both for the
    one-warp-per-solve kernel with express lanes and for the stage-task kernel, whose dispatch order is the counting sort of the
    per-instance costs and histogram the exact cycle left."""
    from wbc_quadruped_dob_b200 import api
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=23)
    a = api.WbcBatch(max_batch=n, device=0)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        for exact in (False, True):
            a.set_observer_state(sc["obs_yd"], sc["obs_yw"])
            a.cycle(sc, exact=exact)
        yd, yw = a.get_observer_state(n)
        last = a.cycle(sc)
        b.set_observer_state(yd, yw)
        fresh = b.cycle(sc)
        for k in fresh:
            assert np.array_equal(last[k], fresh[k]), k
        a.solver_shape()
        assert a.last_solver_kernel == kernel
    finally:
        a.close()
        b.close()


def test_invalid_inputs_and_hold_tau(gpu_batch):
    from wbc_quadruped_dob_b200 import api
    n = 64
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), seed=24)
    bad = dict(sc)
    bad["mode"] = sc["mode"].copy(); bad["mode"][3] = 7
    bad["q"] = sc["q"].copy(); bad["q"][2, 5] = np.nan
    res = {}
    for exact in (False, True):
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        res[exact] = gpu_batch.cycle(bad, exact=exact)
    for k in ("tau", "w"):
        ok = np.ones(n, bool); ok[[3, 5]] = False
        assert np.array_equal(res[True][k][:, ~ok], res[False][k][:, ~ok], equal_nan=True)
    assert res[True]["status"][3] == -20 and res[True]["status"][5] == -21
    assert not res[True]["x"][:, [3, 5]].any()
    p = api.default_params()
    p.hold_tau_on_failure = 1
    gpu_batch.set_params(p)
    try:
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        good = gpu_batch.cycle(sc, exact=True)
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        held = gpu_batch.cycle(bad, exact=True)
    finally:
        gpu_batch.set_params(api.default_params())
    assert np.array_equal(held["tau"][:, [3, 5]], good["tau"][:, [3, 5]])


def test_device_path_equals_host_path(gpu_batch):
    import torch
    n = 1024
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=25)
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    host = gpu_batch.cycle(sc, exact=True)
    dev = torch.device("cuda", 0)
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray) and k != "mode" and not k.startswith("obs")}
    din["mode"] = torch.from_numpy(np.ascontiguousarray(sc["mode"], dtype=np.int32)).to(dev)
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "x": torch.zeros(30, n, dtype=torch.float64, device=dev), "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    gpu_batch.cycle_device(din, dout, n, n, exact=True)
    for k in ("tau", "w", "x", "status"):
        assert np.array_equal(dout[k].cpu().numpy(), host[k]), k


def test_closed_loop_trot_exact_mode(gpu_batch):
    """4 096 robots trotting in place through the forward-dynamics plant (test_fdyn_plant.py's loop, 320 cycles, pushes) with
    every QP solved exactly: no solve fails and every robot stays up."""
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
    diag = torch.zeros(2, n, dtype=torch.float64, device=dev)
    gpu_batch.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    fails, anchor = 0, None
    for c in range(8 * P):
        mode = sched[(c // P) % 4]
        if c % P == 0:
            host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
            _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
            din["mode"] = torch.full((n,), mode, dtype=torch.int32, device=dev)
        sp, sv, sa = trot_in_place_targets(anchor, mode, (c % P) / P, P * 0.0025, height)
        din["sw_des_pos"].copy_(torch.from_numpy(sp)); din["sw_des_vel"].copy_(torch.from_numpy(sv)); din["sw_des_acc"].copy_(torch.from_numpy(sa))
        gpu_batch.cycle_device(din, dout, n, n, exact=True)
        fails += int((dout["status"] != 0).sum().item())
        gpu_batch.plant_dynamics_step(din, dout["tau"], dpush if P <= c < 3 * P else zero, n=n, ld=n, substeps=5, gamma=100.0, diag=diag)
    pos = din["base_pos"].cpu().numpy()
    rpy = din["base_rpy"].cpu().numpy()
    print("closed-loop trot, exact mode: %d robots x %d cycles, failed solves %d, max |base drift| %.1f mm"
          % (n, 8 * P, fails, 1e3 * np.abs(pos - base0).max()))
    assert fails == 0
    assert np.abs(pos - base0).max() < 0.08 and np.abs(rpy - sc["base_rpy"]).max() < 0.15
