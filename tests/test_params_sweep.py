"""The control cycle away from default_params(): every wbc_params field of the controller, changed alone and all at once, against
the oracle run with the same parameters, on the host emulation and on the GPU.

Every kernel takes its gains, weights and limits from `Params P` by value, read in many places: the estimate, Wcom_des, the
joint-limit rows, the swing PD and the friction rows (wbc_front.cuh, wbc_front_leg.cuh), Q, c, the objective and the torque
rows (wbc_assemble.cuh), the momentum plant (wbc_b200.cu) and the forward-dynamics plant (wbc_front.cuh).  A lane that reads the
wrong field, or a constant equal to the default, passes every test that runs at the defaults; the tests here do not.

PLAN pairs each field with a scenario in which it moves the torques (the sensitivity guard checks that it does):
  * kcom, dcom, g_acc, obs_gain, obs_dt, gravity and every field at once: S.make, mixed modes, pushes;
  * q1_weight, slack_weight, kp_sw, kd_sw: swing modes (the slack variables and the swing PD exist only there);
  * mu: stance, terrain off (with terrain the frames' own mu replaces P.mu);
  * joint_dt, tau_max: near_limit (tests/test_qp_limits.py), where joint-limit and torque rows bind.  In S.make's scenarios no
    joint-limit row is active and joint_dt moves no torque at all.
Near the limits DENSE-AUL stops on its iteration count and rounding decides its result (test_qp_limits.py), so there the cycle
is checked in exact mode against the certified optimum x* of the QPs the oracle assembles with the same parameters, with
test_qp_limits.py's rule: within 1e-9 of x*, and WBC_ST_INFEASIBLE exactly where the feasibility LP finds no point.  EDGES
are checked in exact mode only.

Measured on the host emulation (g++ -ffp-contract=off), 200 robots per scenario, seed 5: every perturbation outside the
near-limit scenario within 5e-10 relative torque error of the live oracle; the guard's floors sit at about half of the
measured shares.
"""
import ctypes as C
import os

import numpy as np
import pytest

from tests import qp_exact as E
from tests import qp_exact_lp as LP
from tests import util
from tests.test_qp_dual import DualEmu
from tests.test_qp_limits import ST_INFEASIBLE, near_limit, row_families
from wbc_quadruped_dob_b200 import scenarios as S

GRAVITY = (0.0, 0.0, -9.8)
MIX = {"mixed": (0.34, 0.33, 0.33), "swing": (0.0, 0.5, 0.5), "stance": (1.0, 0.0, 0.0)}

# (field, value, scenario, moved, share): the guard asks the emulated torques to move by more than `moved` (relative to the
# instance's largest torque) on at least `share` of the instances, against the default cycle.  Measured shares (200 robots):
# kcom, dcom, g_acc, obs_gain, obs_dt, q1_weight, kp_sw, kd_sw and all at once 1.0 above 1e-3; slack_weight 1e4 1.0 above 1e-6
# (median 2.3e-4), 1e12 1.0 above 1e-9 (median 2.3e-8: the slack is already ~0 at 1e8); mu 0.3 / 0.9 0.965 / 0.875; joint_dt
# 0.01 / 0.05 0.985 / 0.975; tau_max 40 / 90 0.78 / 0.595; gravity 0.275 / 0.315 (stance instances only: no swing torque moves,
# in the oracle as in the emulation).
PLAN = [("kcom", 1500.0, "mixed", 1e-3, 0.5), ("kcom", 4000.0, "mixed", 1e-3, 0.5),
        ("dcom", 20.0, "mixed", 1e-3, 0.5), ("dcom", 90.0, "mixed", 1e-3, 0.5),
        ("g_acc", 9.5, "mixed", 1e-3, 0.5), ("g_acc", 10.2, "mixed", 1e-3, 0.5),
        ("obs_gain", 4.0, "mixed", 1e-3, 0.5), ("obs_gain", 40.0, "mixed", 1e-3, 0.5),
        ("obs_dt", 0.001, "mixed", 1e-3, 0.5), ("obs_dt", 0.005, "mixed", 1e-3, 0.5),
        ("q1_weight", 10.0, "swing", 1e-3, 0.5), ("q1_weight", 200.0, "swing", 1e-3, 0.5),
        ("slack_weight", 1e4, "swing", 1e-6, 0.5), ("slack_weight", 1e12, "swing", 1e-9, 0.5),
        ("kp_sw", 150.0, "swing", 1e-3, 0.5), ("kp_sw", 600.0, "swing", 1e-3, 0.5),
        ("kd_sw", 8.0, "swing", 1e-3, 0.5), ("kd_sw", 45.0, "swing", 1e-3, 0.5),
        ("mu", 0.3, "stance", 1e-3, 0.45), ("mu", 0.9, "stance", 1e-3, 0.4),
        ("joint_dt", 0.01, "limit", 1e-3, 0.45), ("joint_dt", 0.05, "limit", 1e-3, 0.45),
        ("tau_max", 40.0, "limit", 1e-3, 0.35), ("tau_max", 90.0, "limit", 1e-3, 0.3),
        ("gravity", (0.3, -0.2, -9.7), "mixed", 1e-3, 0.12), ("gravity", (0.0, 0.0, -10.5), "mixed", 1e-3, 0.12),
        ("all", dict(kcom=3000.0, dcom=40.0, q1_weight=80.0, slack_weight=1e6, mu=0.5, tau_max=70.0, joint_dt=0.03, kp_sw=400.0,
                     kd_sw=25.0, g_acc=9.7, obs_gain=15.0, obs_dt=0.003, gravity=(0.2, 0.1, -9.9)), "mixed", 1e-3, 0.5)]
# exact mode only: mu = 0 (the pyramid collapses to tangential force 0), a joint_dt that scales the joint-limit rows by
# 2 / dt^2 = 2e6, slack_weight = 1, a tau_max no torque row can reach
EDGES = [("mu", 0.0, "stance"), ("joint_dt", 1e-3, "limit"), ("slack_weight", 1.0, "swing"), ("tau_max", 1e6, "limit")]


def pid(e):
    return "%s=%s" % (e[0], "" if e[0] == "all" else ("%g,%g,%g" % e[1] if e[0] == "gravity" else "%g" % e[1]))


def changes(field, value):
    return dict(value) if field == "all" else {field: value}


def apply(p, ch):
    """Set the fields of `ch` on a Params struct (api.Params, util.EmuParams or the oracle's, which has no gravity)."""
    for k, v in ch.items():
        if k != "gravity":
            setattr(p, k, v)
        elif hasattr(p, "gravity"):
            p.gravity[:] = v
    return p


def oracle_args(oracle, ch):
    return dict(params=apply(oracle.default_params(), ch), gravity=ch.get("gravity", GRAVITY))


def scenario(kind, n, seed):
    return near_limit(n, seed=seed) if kind == "limit" else S.make(n, mode_mix=MIX[kind], pushes=True, seed=seed)


def oracle_qps(oracle, sc, idx, w, ch):
    """The QPs the oracle assembles for instances idx with the parameters `ch` and the observer wrenches w [6, n]."""
    kw = oracle_args(oracle, ch)
    out = []
    for i in idx:
        _, qp = oracle.assemble_only(sc, int(i), w=w[:, i], **kw)
        out.append((np.array(qp.Q).reshape(30, 30), np.array(qp.c), np.array(qp.L)[:qp.nrows * 31].reshape(qp.nrows, 31), qp.neq))
    return out


# The feasibility LP's margin |t*| (row-scaled) must stay clear of 0 wherever it decides, so that no decision rests on a
# tolerance (test_qp_limits.py's floor).  Measured on the host and B200 batches: at least 1.6e-3 (joint_dt = 1e-3; 4.7e-3 otherwise).
LP_MARGIN_FLOOR = 1e-4


def check_exact(what, qps, x, status, decide_by_lp):
    """Exact-mode x [n, 30] and status against x*: within 1e-9 of the certified optimum; with decide_by_lp, WBC_ST_INFEASIBLE
    (x = 0) exactly where the feasibility LP finds no point, otherwise status 0 on every QP.  Returns the worst error."""
    if decide_by_lp:
        t = np.array([LP.lp_margin(L, neq)[0] for _, _, L, neq in qps])
        print("%s: feasibility LP, smallest |t*| %.3e" % (what, np.abs(t).min()))
        assert np.abs(t).min() >= LP_MARGIN_FLOOR, (what, "the LP margin is too close to 0 to decide feasibility")
        feas = t <= 0.0
        assert np.array_equal(status == 0, feas), what
    else:
        feas = status == 0
        assert feas.all(), (what, "refused", np.flatnonzero(~feas), status[~feas])
    assert (status[~feas] == ST_INFEASIBLE).all() and not x[~feas].any(), what
    e = np.array([E.err(x[k], LP.certified_qp(*qps[k], x0=x[k])[0]) for k in np.flatnonzero(feas)])
    print("%s: worst x* err %.3e over %d feasible, %d infeasible" % (what, e.max(), feas.sum(), (~feas).sum()))
    assert e.max() <= 1e-9, what
    return e.max()


def check_no_tangential_force(what, x):
    """mu = 0, stance: the tangential components of the four contact forces x[18:30] are zero (to 1e-9 of the largest |x|)."""
    ft = np.hstack([x[:, [18 + 3 * f, 19 + 3 * f]] for f in range(4)])
    print("%s, mu = 0: largest tangential force %.3e N" % (what, np.abs(ft).max()))
    assert np.abs(ft).max() <= 1e-9 * max(1.0, np.abs(x).max()), what


# ---------------------------------------------------------------------------------------------------------------------
# host emulation

N_CPU = 200
SEED_CPU = 5


@pytest.fixture(scope="module")
def cpu_scenarios():
    return {k: scenario(k, N_CPU, SEED_CPU) for k in ("mixed", "swing", "stance", "limit")}


@pytest.fixture(scope="module")
def default_cycles(emu, cpu_scenarios):
    return {k: emu.cycle(sc) for k, sc in cpu_scenarios.items()}


@pytest.fixture(scope="module")
def dual():
    return DualEmu()


def emu_exact_cycle(emu, dual, sc, P):
    """The emulated front end with parameters P, then the device's assembly (assemble_qp) and the exact solver (qp_dual.cuh) on
    each record: (front outputs, x [n, 30], status [n])."""
    out = emu.cycle(sc, params=P)
    n = out["rec"].shape[0]
    emu.lib.emu_assemble.argtypes = [C.POINTER(util.EmuParams)] + [C.POINTER(C.c_double)] * 4 + [C.POINTER(C.c_int)] * 2
    x, status = np.zeros((n, 30)), np.zeros(n, np.int32)
    Q, c, L = np.zeros(900), np.zeros(30), np.zeros(86 * 31)
    nrows, neq = C.c_int(), C.c_int()
    d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    for i in range(n):
        rec = np.ascontiguousarray(out["rec"][i])
        emu.lib.emu_assemble(C.byref(P), d(rec), d(Q), d(c), d(L), C.byref(nrows), C.byref(neq))
        x[i], status[i] = dual.solve(Q.reshape(30, 30), c, L[:nrows.value * 31].reshape(nrows.value, 31), neq.value)[:2]
    return out, x, status


@pytest.mark.parametrize("entry", PLAN, ids=pid)
def test_sensitivity_guard(emu, cpu_scenarios, default_cycles, entry):
    """Each perturbation moves the emulated torques in its scenario: a plan that drifts into a regime where its field does
    nothing fails here instead of passing the parity tests without testing anything."""
    field, value, kind, moved, share = entry
    got = emu.cycle(cpu_scenarios[kind], params=apply(util.emu_default_params(), changes(field, value)))
    d = util.rel_rows(got["tau"].T, default_cycles[kind]["tau"].T)
    print("%s on %s: torques moved by more than %.0e on %.3f of the instances (median %.2e)" % (pid(entry), kind, moved, (d > moved).mean(),
                                                                                             np.median(d)))
    assert (d > moved).mean() >= share


@pytest.mark.parametrize("entry", [e for e in PLAN if e[2] != "limit"], ids=pid)
def test_emulation_matches_oracle(emu, oracle, oracle_qp, cpu_scenarios, entry):
    """The emulated cycle against the live oracle run with the same parameters and gravity: util.check_cycle_parity's
    tolerances, and the observer state it leaves."""
    field, value, kind = entry[:3]
    ch = changes(field, value)
    sc = cpu_scenarios[kind]
    got = emu.cycle(sc, params=apply(util.emu_default_params(), ch))
    ref, _ = oracle.run_cycle_batch(sc, nthreads=8, solver=oracle_qp, **oracle_args(oracle, ch))
    worst = util.check_cycle_parity(got, ref, what=pid(entry))
    for k in ("yd", "yw"):
        assert np.abs(got[k].T - ref[k]).max() <= util.TOL_OBS * max(1.0, np.abs(ref[k]).max()), k
    print("%s: worst torque rel err %.3e" % (pid(entry), worst))


EXACT_CPU = [e[:3] for e in PLAN if e[2] == "limit" or e[0] in ("mu", "slack_weight", "all")] + EDGES


@pytest.mark.parametrize("entry", EXACT_CPU, ids=pid)
def test_exact_emulation_matches_certified_optimum(emu, oracle, dual, cpu_scenarios, entry):
    """Exact mode on the host: the emulated front end and assembly with the perturbed parameters, solved by the exact solver's
    emulation, against x* of the QPs the oracle assembles with the same parameters (and the emulation's observer wrench).
    Near the limits feasibility is decided by the LP (its margin checked against LP_MARGIN_FLOOR).

    mu = 0: every tangential row comes with its negation, so the feasible set has no interior (the LP margin is exactly 0)
    and every QP is feasible with the tangential forces zero.  Every one must be solved, at x*, with those forces zero: the
    exact solver holds out the second row of a pair when rounding shows it violated after the first joined the active set
    (qp_dual.cuh, TOL_HOLD; before that, 2 of these 200 QPs were refused as infeasible)."""
    field, value, kind = entry
    ch = changes(field, value)
    sc = cpu_scenarios[kind]
    out, x, status = emu_exact_cycle(emu, dual, sc, apply(util.emu_default_params(), ch))
    qps = oracle_qps(oracle, sc, range(N_CPU), out["w"], ch)
    edge = (field, value, kind) in EDGES
    check_exact("exact emulation %s%s" % (pid(entry), " (edge)" if edge else ""), qps, x, status, kind == "limit")
    if (field, value) == ("mu", 0.0):
        check_no_tangential_force("exact emulation", x)
    if (field, value) == ("tau_max", 1e6):
        for k in np.flatnonzero(status == 0):
            Q, c, L, neq = qps[k]
            tq, _ = row_families(L.shape[0], neq)
            assert (L[tq, :30] @ x[k] - L[tq, 30]).max() < -1e5, k          # no torque row is anywhere near binding


GRAVITIES = [(0.3, -0.2, -9.7), (0.0, 0.0, -10.5)]
FDYN = [dict(obs_dt=0.001), dict(obs_dt=0.005), dict(gravity=GRAVITIES[0]), dict(gravity=GRAVITIES[1]),
        dict(obs_dt=0.004, gravity=(-0.25, 0.4, -9.6))]


def fdyn_inputs(n, seed):
    sc = S.make(n, mode_mix=MIX["mixed"], pushes=False, seed=seed)
    rng = np.random.default_rng(seed)
    return sc, rng.normal(0.0, 4.0, (12, n)), rng.normal(0.0, 15.0, (6, n))


def check_fdyn(what, got, ref, base):
    for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq"):
        assert np.abs(got[k] - ref[k]).max() <= 1e-9 * max(1.0, np.abs(ref[k]).max()), (what, k)
    assert np.abs(got["foot_force"] - ref["foot_force"]).max() <= 1e-8 * max(1.0, np.abs(ref["foot_force"]).max()), what
    moved = np.abs(got["base_vel"] - base["base_vel"]).max()
    print("%s: base velocity moved by %.3e against the default parameters" % (what, moved))
    assert moved > 1e-4, what


@pytest.mark.parametrize("ch", FDYN, ids=lambda ch: ",".join("%s=%s" % kv for kv in ch.items()))
def test_fdyn_plant_emulation_off_defaults(emu, oracle, ch):
    """The forward-dynamics plant (fdyn_step_instance, compiled for the host) with a non-default control period and gravity
    against the oracle's dense formulation, with test_fdyn_plant.py's tolerances."""
    sc, tau, push = fdyn_inputs(48, 17)
    base, _ = emu.fdyn_step(sc, tau, push, nsub=5, gamma=100.0)
    got, _ = emu.fdyn_step(sc, tau, push, nsub=5, gamma=100.0, params=apply(util.emu_default_params(), ch))
    ref, _ = oracle.fdyn_step(sc, tau, push, nsub=5, gamma=100.0, **oracle_args(oracle, ch))
    check_fdyn("emulated dynamics plant %s" % ch, got, ref, base)


# ---------------------------------------------------------------------------------------------------------------------
# the CUDA kernels

N_GPU = 2048
N_GPU_LIMIT = 1024
SEED_GPU = 31
EVERY = 16              # exact mode: x* certified on every EVERY-th instance
# Default mode near the limits, against the emulation: DENSE-AUL stops there on its iteration count at a large penalty and
# amplifies rounding (test_qp_limits.TOL_X_SAME), so an instance either takes the emulation's decisions (same Cholesky count,
# x within TOL_X_SAME) or not, and a share of them must.  Measured on a B200, 1 024 robots: 96.9 % to 98.4 % of the instances
# have equal counts; where they do, x is within 1.3e-4 of the emulation's, and within 6.8e-4 for tau_max = 90 on the four-lane
# front kernel; both hold on at least 96.7 % of the instances.  A field read wrongly moves every instance whose torque or joint-limit rows bind (35-98 % here, the
# sensitivity guard) by O(1).
NEAR_LIMIT_AGREE = 0.95


def _ctx(n, params=None, **env):
    """A ctx created with the environment variables `env` set (the library reads them at wbc_create); the caller's environment
    is restored afterwards."""
    from wbc_quadruped_dob_b200 import api
    saved = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return api.WbcBatch(max_batch=n, device=0, params=params)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def gpu_params(ch):
    from wbc_quadruped_dob_b200 import api
    return apply(api.default_params(), ch)


@pytest.fixture(scope="module")
def fronts():
    """One ctx per front kernel: the four-lane one (the default) and the thread-per-instance one (WBC_FRONT=thread)."""
    ctxs = {"leg": _ctx(N_GPU), "thread": _ctx(N_GPU, WBC_FRONT="thread")}
    yield ctxs
    for b in ctxs.values():
        b.close()


def _cycle(b, sc, **kw):
    b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    return b.cycle(sc, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", [e[:3] for e in PLAN] + EDGES, ids=pid)
def test_gpu_cycle_off_defaults(fronts, emu, oracle, oracle_qp, entry):
    """wbc_cycle with the perturbed parameters set on a live ctx, both front kernels, default and exact mode.
    Default mode: against the live oracle (util.check_cycle_parity); near the limits against the emulation (status equal, the
    emulation's decisions on NEAR_LIMIT_AGREE of the instances).  Exact mode: x within 1e-9 of x* on every EVERY-th instance,
    WBC_ST_INFEASIBLE exactly where the LP finds no point, status 0 on the whole batch elsewhere.  mu = 0: every instance of the
    batch solved, at x* with zero tangential forces."""
    from tests.test_qp_limits import TOL_X_SAME
    from wbc_quadruped_dob_b200 import api
    field, value, kind = entry
    ch = changes(field, value)
    edge = entry in EDGES
    n = N_GPU_LIMIT if kind == "limit" else N_GPU
    sc = scenario(kind, n, SEED_GPU)
    if kind == "limit":
        ref = emu.cycle(sc, params=apply(util.emu_default_params(), ch))
    elif not edge:
        ref, _ = oracle.run_cycle_batch(sc, nthreads=os.cpu_count(), solver=oracle_qp, **oracle_args(oracle, ch))
    idx = np.arange(0, n, EVERY)
    for front, b in fronts.items():
        b.set_params(gpu_params(ch))
        try:
            got = _cycle(b, sc) if not edge else None
            ex = _cycle(b, sc, exact=True)
        finally:
            b.set_params(api.default_params())
        what = "GPU %s front %s" % (front, pid(entry))
        if kind == "limit" and not edge:
            same = got["qp_info"][0] == ref["qp_info"][0]
            rel = np.abs(got["x"] - ref["x"]).max(axis=0) / np.maximum(1.0, np.abs(ref["x"]).max(axis=0))
            agree = same & (rel <= TOL_X_SAME)
            print("%s: default mode, ncholesky equal to the emulation's on %.4f, worst x distance there %.3e, both on %.4f"
                  % (what, same.mean(), rel[same].max(), agree.mean()))
            assert np.array_equal(got["status"], ref["status"]) and agree.mean() >= NEAR_LIMIT_AGREE, what
        elif not edge:
            print("%s: default mode, worst torque rel err %.3e" % (what, util.check_cycle_parity(got, ref, what=what)))
        if kind != "limit":
            assert (ex["status"] == 0).all(), (what, "refused", np.flatnonzero(ex["status"]))
        sub = np.arange(n) if (field, value) == ("mu", 0.0) else idx
        qps = oracle_qps(oracle, sc, sub, ex["w"], ch)
        check_exact(what + " exact", qps, ex["x"][:, sub].T, ex["status"][sub], kind == "limit")
        if (field, value) == ("mu", 0.0):
            check_no_tangential_force(what, ex["x"].T)


STAGED = [("q1_weight", 200.0, "swing"), ("slack_weight", 1e4, "swing"), ("tau_max", 40.0, "limit"), PLAN[-1][:3]]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", STAGED, ids=pid)
def test_gpu_staged_solver_off_defaults(oracle, oracle_qp, entry):
    """The stage-task solver kernel (a batch of 49 152 >= WBC_STAGED_MIN_N) with the perturbed parameters given at wbc_create:
    bit for bit the one-warp-per-solve kernel (WBC_SOLVER=mono) on the same batch, and outside the near-limit scenario every
    64th instance against the live oracle."""
    field, value, kind = entry
    ch = changes(field, value)
    n = 49152
    sc = scenario(kind, n, SEED_GPU + 1)
    res = {}
    for solver in ("staged", "mono"):
        b = _ctx(n, params=gpu_params(ch), WBC_SOLVER=solver)
        try:
            o = _cycle(b, sc)
            b.solver_shape()
            res[solver] = (o, b.last_solver_kernel)
        finally:
            b.close()
    (o1, k1), (o2, k2) = res["staged"], res["mono"]
    assert (k1, k2) == ("wbc_solve_staged_kernel", "wbc_solve_kernel")
    for k in o1:
        assert np.array_equal(o1[k], o2[k]), k
    if kind != "limit":
        idx = np.arange(0, n, 64)
        sub = {k: (np.ascontiguousarray(v[..., idx]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
        ref, _ = oracle.run_cycle_batch(sub, nthreads=os.cpu_count(), solver=oracle_qp, **oracle_args(oracle, ch))
        got = {k: v[..., idx] for k, v in o1.items()}
        print("GPU staged %s: worst torque rel err %.3e" % (pid(entry), util.check_cycle_parity(got, ref, what=pid(entry))))


@pytest.mark.gpu
@pytest.mark.parametrize("g", GRAVITIES, ids=lambda g: "%g,%g,%g" % g)
def test_gpu_debug_update_with_gravity(fronts, oracle, g):
    """wbc_debug_update with a non-default gravity vector against oracle.update_only with the same one, with the tolerances of
    test_gpu_parity.test_update_stages_match_oracle; the gravity terms must differ from those of the default vector."""
    from wbc_quadruped_dob_b200 import api
    b = fronts["leg"]
    sc = S.make(64, mode_mix=MIX["mixed"], pushes=True, seed=77)
    b.set_params(gpu_params({"gravity": g}))
    try:
        dbg = b.debug_update(sc)
    finally:
        b.set_params(api.default_params())
    tol = dict(M=1e-12, h=1e-11, g=1e-11, Jac_lin=1e-13, Jdqd_lin=1e-12, com=1e-13, com_vel=1e-13, hcom=1e-11, gcom=1e-11,
               Jcom_lin=1e-13, Jdqdcom_lin=1e-12, foot_pos=1e-13, foot_vel=1e-13)
    for i in range(0, 64, 7):
        d = oracle.update_only(sc, i, gravity=g)
        for k, t in tol.items():
            assert np.abs(dbg[k][:, i] - np.array(getattr(d, k))).max() < t, (i, k)
        assert np.abs(dbg["g"][:, i] - np.array(oracle.update_only(sc, i).g)).max() > 1e-2
        Mcom = np.array(d.Mcom).reshape(18, 18)
        assert np.abs(dbg["Mcom_b"][:, i].reshape(6, 6) - Mcom[:6, :6]).max() < 1e-12
        assert np.abs(dbg["Mcom_j"][:, i].reshape(12, 12) - Mcom[6:, 6:]).max() < 1e-13


LIVE = [("kcom", 4000.0, "mixed"), ("q1_weight", 10.0, "swing"), ("mu", 0.3, "stance"), ("joint_dt", 0.01, "limit"),
        ("tau_max", 40.0, "limit"), ("gravity", GRAVITIES[0], "mixed"), PLAN[-1][:3]]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", LIVE, ids=pid)
def test_gpu_params_changed_on_a_live_context(entry):
    """One ctx runs default -> perturbed -> default on 4 096 robots (express lanes on, longest-first dispatch from the second
    cycle on): the perturbed cycle is bit for bit a fresh ctx created with those parameters, and the last one bit for bit the
    ctx's first, fresh, default cycle.  A parameter change takes effect on the next cycle and leaves nothing behind in the
    dispatch state."""
    from wbc_quadruped_dob_b200 import api
    field, value, kind = entry
    p = gpu_params(changes(field, value))
    n = 4096
    sc = scenario(kind, n, SEED_GPU + 2)
    live, fresh = _ctx(n), _ctx(n, params=p)
    try:
        first = _cycle(live, sc)
        live.set_params(p)
        pert = _cycle(live, sc)
        live.set_params(api.default_params())
        last = _cycle(live, sc)
        want = _cycle(fresh, sc)
    finally:
        live.close()
        fresh.close()
    assert not np.array_equal(pert["tau"], first["tau"])
    for k in want:
        assert np.array_equal(pert[k], want[k]), ("perturbed", k)
        assert np.array_equal(last[k], first[k]), ("back to default", k)


WARM = [("tau_max", 40.0, "limit"), ("mu", 0.3, "stance")]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", WARM, ids=pid)
def test_gpu_warm_sets_across_a_parameter_change(oracle, entry):
    """Warm exact mode on one ctx, default -> perturbed -> default: the active sets stored under one tau_max or mu start the
    next cycle under another, and every cycle still gives x* (every EVERY-th instance, the LP deciding feasibility near the
    limits), with the instances warm-started where the previous cycle stored a set."""
    from wbc_quadruped_dob_b200 import api
    field, value, kind = entry
    n = 2048
    sc = scenario(kind, n, SEED_GPU + 3)
    idx = np.arange(0, n, EVERY)
    b = _ctx(n)
    try:
        for k, ch in enumerate(({}, {field: value}, {})):
            b.set_params(gpu_params(ch))
            got = _cycle(b, sc, exact=True, warm=True)
            started = (got["qp_info"][5] & api.FL_WARM_STARTED) != 0
            if k:
                assert started[prev == 0].all() and not started[prev != 0].any()
            prev = got["status"].copy()
            qps = oracle_qps(oracle, sc, idx, got["w"], ch)
            check_exact("GPU warm cycle %d (%s)" % (k, pid(entry) if ch else "default"), qps, got["x"][:, idx].T, got["status"][idx],
                        kind == "limit")
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ch", FDYN, ids=lambda ch: ",".join("%s=%s" % kv for kv in ch.items()))
def test_gpu_fdyn_plant_off_defaults(fronts, oracle, ch):
    """wbc_plant_dynamics_step with the ctx's control period and gravity off their defaults against oracle.fdyn_step."""
    from wbc_quadruped_dob_b200 import api
    sc, tau, push = fdyn_inputs(200, 18)
    b = fronts["leg"]
    out = {}
    for key, c in (("base", {}), ("got", ch)):
        st = {k: np.array(sc[k], dtype=np.float64, order="C") for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
        st["foot_force"] = np.zeros((12, 200)); st["mode"] = np.ascontiguousarray(sc["mode"], dtype=np.int32)
        b.set_params(gpu_params(c))
        try:
            b.plant_dynamics_step(st, tau, push, substeps=5, gamma=100.0)
        finally:
            b.set_params(api.default_params())
        out[key] = st
    ref, _ = oracle.fdyn_step(sc, tau, push, nsub=5, gamma=100.0, **oracle_args(oracle, ch))
    check_fdyn("GPU dynamics plant %s" % ch, out["got"], ref, out["base"])


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [dict(obs_dt=0.001), dict(obs_dt=0.005), dict(g_acc=9.5), dict(g_acc=10.2), dict(obs_dt=0.004, g_acc=9.7)],
                         ids=lambda ch: ",".join("%s=%g" % kv for kv in ch.items()))
def test_gpu_momentum_plant_off_defaults(fronts, oracle, oracle_qp, ch):
    """wbc_plant_step (the momentum plant of the push sweep) after a cycle with non-default obs_dt and g_acc, closed through the
    commanded forces and open loop, against oracle.plant_step with the same parameters (test_push_sweep.py's tolerances).  GPU
    only: the plant is a kernel of wbc_b200.cu, which the host emulation does not build (the record fields it reads come from
    the front end, which the emulation tests above cover off the defaults)."""
    from wbc_quadruped_dob_b200 import api
    n = 512
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=True, seed=SEED_GPU + 4)
    push = np.random.default_rng(4).normal(0.0, 30.0, (6, n))
    b = fronts["leg"]
    b.set_params(gpu_params(ch))
    try:
        got = _cycle(b, sc)
        pos, vel, ff = sc["base_pos"].copy(), sc["base_vel"].copy(), sc["foot_force"].copy()
        b.plant_step(pos, vel, push, foot_force=ff, x=got["x"])
        opos, ovel = sc["base_pos"].copy(), sc["base_vel"].copy()
        b.plant_step(opos, ovel, push)
    finally:
        b.set_params(api.default_params())
    kw = oracle_args(oracle, ch)
    ref, _ = oracle.run_cycle_batch(sc, nthreads=os.cpu_count(), solver=oracle_qp, **kw)
    util.check_cycle_parity(got, ref, what="momentum plant cycle %s" % ch)
    rpos, rvel, rff = oracle.plant_step(sc, push, x=got["x"].T, **kw)
    assert np.abs(vel - rvel).max() <= 1e-10 and np.abs(pos - rpos).max() <= 1e-12
    assert np.abs(ff - rff).max() <= 1e-10 * max(1.0, np.abs(rff).max())
    rpos, rvel, _ = oracle.plant_step(sc, push, **kw)
    assert np.abs(ovel - rvel).max() <= 1e-10 and np.abs(opos - rpos).max() <= 1e-12
    dpos, dvel, _ = oracle.plant_step(sc, push, params=oracle.default_params())
    print("momentum plant %s: base velocity moved by %.3e against the default parameters" % (ch, np.abs(rvel - dvel).max()))
    assert np.abs(rvel - dvel).max() > 1e-4
