"""SURVEY.md 8f-3: the observer forms of the reference's dead ESTIMATOR_SEM (dogbot_controller/src/client/estimator_sem.cpp:24-106) --
explicit gain, second-order recursion through `ygamma`, and the foot-wrench map getw3 -- device code against the oracle.

PARITY UNPINNED: the reference never calls ESTIMATOR_SEM (SURVEY.md 2, row 4) and holds no vectors for it; the oracle restates
estimator_sem.cpp's lines, numpy's pinv is the pseudo-inverse getw3 takes from Eigen, and the recursions are also checked against
their closed-form responses.  CPU tests run the device headers through the host emulation; GPU tests go through the C ABI.

The chained-cycle tests run the oracle with the `oracle_qp` fixture's QP solver (the restatement where the reference ALGLIB is not
built): what they check is the observer and how its estimate enters the QP and the torques, not the solve."""
import numpy as np
import pytest

from oracle import oracle_py as O
from tests import util
from wbc_quadruped_dob_b200 import scenarios as S

FORMS = [(1, 1), (2, 0), (2, 1)]      # (order, form); (1, 0) is DOGCTRL::estimate(), covered by the parity tests


def _params(order, form, k2=4.0, emu=False):
    if emu:
        p = util.emu_default_params()
    else:
        from wbc_quadruped_dob_b200 import api
        p = api.default_params()
    p.obs_order, p.obs_form, p.obs_gain2 = order, form, k2
    return p


def _oracle_params(order, form, k2=4.0):
    p = O.default_params()
    p.obs_order, p.obs_form, p.obs_gain2 = order, form, k2
    return p


def test_second_order_recursion_has_the_closed_form_response():
    """Constant disturbance into the recursion alone (rho - int(d) = w_true t): the estimate follows the step response of
    k1 k2 / (s^2 + k2 s + k1 k2) -- for k1 = 10, k2 = 50 an over-damped pair -- and settles on w_true."""
    k1, k2, T, w_true = 10.0, 50.0, 0.0025, 3.0
    for form in (0, 1):
        yw = yg = 0.0
        hist = []
        for k in range(1, 1601):
            e = w_true * T * k - yw                 # rho - yd - yw_prev with rho - yd = integral of the true disturbance
            if form == 0:
                w = k2 * (yg + T * k1 * e) / (1.0 + k2 * T + k1 * k2 * T * T)
                yg = yg + T * (k1 * (e - w * T) - w)
            else:
                yg = yg + T * (k1 * e - k2 * yg)
                w = k2 * yg
            yw += w * T
            hist.append(w)
        t = T * np.arange(1, 1601)
        s1, s2 = np.roots([1.0, k2, k1 * k2])
        exact = w_true * (1.0 + (s2 * np.exp(s1 * t) - s1 * np.exp(s2 * t)) / (s1 - s2)).real
        assert abs(hist[-1] - w_true) < 1e-6 * w_true
        assert np.max(np.abs(np.array(hist) - exact)) < 0.03 * w_true      # first-order integrators, T k2 = 0.125


@pytest.mark.parametrize("order,form", FORMS)
def test_emulated_device_code_matches_the_oracle_over_chained_cycles(order, form, oracle_qp):
    emu = util.Emu()
    sc = S.make(24, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=False, seed=21)
    sc["obs_yg"] = np.zeros((6, 24))
    pe, po = _params(order, form, emu=True), _oracle_params(order, form)
    rng = np.random.default_rng(5)
    for cyc in range(6):
        ref, _ = O.run_cycle_batch(sc, params=po, solver=oracle_qp)
        got = emu.cycle(sc, params=pe)
        scale = 1.0 + np.abs(ref["w"]).max()
        assert np.max(np.abs(got["w"] - ref["w"].T)) < 1e-9 * scale, (cyc, order, form)
        assert np.max(np.abs(got["yg"] - ref["yg"].T)) < 1e-9 * (1.0 + np.abs(ref["yg"]).max())
        ok = ref["status"] == 0
        tr = ref["tau"].T[:, ok]
        assert np.max(np.abs(got["tau"][:, ok] - tr) / (1.0 + np.abs(tr))) < 1e-6
        # next cycle: carried observer state from the oracle, state nudged so that the momentum changes
        sc["obs_yd"], sc["obs_yw"], sc["obs_yg"] = ref["yd"].T.copy(), ref["yw"].T.copy(), ref["yg"].T.copy()
        sc["base_vel"] = sc["base_vel"] + 0.01 * rng.standard_normal(sc["base_vel"].shape)
        sc["dq"] = sc["dq"] + 0.02 * rng.standard_normal(sc["dq"].shape)
    if order == 2:
        assert np.abs(sc["obs_yg"]).max() > 0.0


def test_emulated_foot_wrench_map_matches_getw3_and_reproduces_the_wrench():
    emu = util.Emu()
    sc = S.make(32, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=False, seed=22)
    sc["obs_yd"] = 0.3 * np.random.default_rng(1).standard_normal((6, 32))      # a non-trivial estimate
    got = emu.cycle(sc)
    for i in range(32):
        dyn = O.update_only(sc, i)
        J = np.array(dyn.Jcom_lin).reshape(12, 18)
        ref = O.foot_wrench_map(J, got["w"][:, i])
        assert np.max(np.abs(got["w3"][:, i] - ref)) < 1e-9 * (1.0 + np.abs(ref).max()), i
        assert np.max(np.abs(J[:, :6].T @ got["w3"][:, i] - got["w"][:, i])) < 1e-9 * (1.0 + np.abs(got["w"][:, i]).max())


@pytest.mark.gpu
@pytest.mark.parametrize("order,form", FORMS)
def test_gpu_observer_forms_match_the_oracle_over_chained_cycles(order, form, oracle_qp):
    from wbc_quadruped_dob_b200 import api
    n = 512
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=False, seed=23)
    sc["obs_yg"] = np.zeros((6, n))
    batch = api.WbcBatch(max_batch=n, params=_params(order, form))
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    po = _oracle_params(order, form)
    rng = np.random.default_rng(6)
    worst_w = worst_tau = 0.0
    for cyc in range(8):
        ref, _ = O.run_cycle_batch(sc, params=po, nthreads=8, solver=oracle_qp)
        got = batch.cycle(sc, want=("status", "w3"))
        worst_w = max(worst_w, float(np.max(np.abs(got["w"] - ref["w"].T)) / (1.0 + np.abs(ref["w"]).max())))
        ok = (ref["status"] == 0) & (got["status"] == 0)
        assert ok.mean() > 0.99
        tr = ref["tau"].T[:, ok]
        worst_tau = max(worst_tau, float(np.max(np.abs(got["tau"][:, ok] - tr) / (1.0 + np.abs(tr)))))
        yd, yw = batch.get_observer_state(n)
        yg = batch.get_observer_state2(n)
        assert np.max(np.abs(yd - ref["yd"].T)) < 1e-9 * (1.0 + np.abs(ref["yd"]).max())
        assert np.max(np.abs(yw - ref["yw"].T)) < 1e-9 * (1.0 + np.abs(ref["yw"]).max())
        if order == 2:
            assert np.max(np.abs(yg - ref["yg"].T)) < 1e-9 * (1.0 + np.abs(ref["yg"]).max())
        sc["obs_yd"], sc["obs_yw"], sc["obs_yg"] = ref["yd"].T.copy(), ref["yw"].T.copy(), ref["yg"].T.copy()
        sc["base_vel"] = sc["base_vel"] + 0.01 * rng.standard_normal(sc["base_vel"].shape)
        sc["dq"] = sc["dq"] + 0.02 * rng.standard_normal(sc["dq"].shape)
    assert worst_w < 1e-9 and worst_tau < 1e-6, (worst_w, worst_tau)


@pytest.mark.gpu
def test_gpu_foot_wrench_map_matches_getw3():
    from wbc_quadruped_dob_b200 import api
    n = 256
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=False, seed=24)
    sc["obs_yd"] = 0.3 * np.random.default_rng(2).standard_normal((6, n))
    batch = api.WbcBatch(max_batch=n)
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    got = batch.cycle(sc, want=("status", "w3"))
    assert np.abs(got["w3"]).max() > 0.0
    for i in range(0, n, 4):
        dyn = O.update_only(sc, i)
        J = np.array(dyn.Jcom_lin).reshape(12, 18)
        ref = O.foot_wrench_map(J, got["w"][:, i])
        assert np.max(np.abs(got["w3"][:, i] - ref)) < 1e-9 * (1.0 + np.abs(ref).max()), i
