"""The controller's QPs where its limits bind: joints at their limits, saturated torques, infeasible rows and spilled working sets.

The scenarios of the other solver tests keep the robot well inside its limits: there the joint-limit rows are never active at
the optimum and the DENSE-AUL working set stays within 13 rows, so several solver paths never run inside a control cycle.  The
batches here (near_limit) put k joints of every robot within `margin` rad of a limit, moving towards it, and reach them:

  * the spill form of the DENSE-AUL solve (qp_warp.cuh, SPILL = true: the working set outgrows NICCAP = 18 and CI, the factor
    and the QQP vectors move to global scratch), in the one-warp kernel and in the stage-task kernel;
  * the literal multiplier update, taken when the reduced one declines (among other cases, past KACAP = 36 active rows);
  * exact mode's WBC_ST_INFEASIBLE on QPs the controller itself assembles.

The reference (tests/qp_exact_lp.py): feasibility is decided by a linear program (lp_margin, scipy's HiGHS), and every
LP-feasible QP gets an optimum certified by qp_exact.certify (certified_qp).  On these QPs qp_exact.exact_qp alone does not
always deliver one: its first phase (add the most violated row) cycles at vertices where more rows than variables meet, or
reaches a singular KKT matrix (from a cold start on 20 of the 882 feasible QPs of the default batch), and its three
refinement steps leave an x 2e-9 from x* at a vertex of nearly dependent rows (multipliers of 3e13, instance 754 of the
exact-mode cycle test below, where the solvers meet the rows to 2e-13).  certified_qp restarts from the LP's point and
refines the final KKT solve ten times.  The LP margin separates the two classes clearly: the smallest |t*| over both
batches is 3.7e-4 (row-scaled), so no decision rests on a solver tolerance.

Measured on the host emulation (g++ -ffp-contract=off), two batches of 1 000 robots (seed 5, default limits; seed 6,
tau_max = 25), observer wrench 0; the counts each test pins are in its docstring.
"""
import numpy as np
import pytest

from tests import qp_exact as E
from tests import qp_exact_lp as P
from tests import util
from tests.test_qp_dual import DualEmu
from tests.test_qp_exact import assemble, by_shape
from wbc_quadruped_dob_b200 import scenarios as S

ST_INFEASIBLE = -22
SPILL, LITERAL = 32, 8                        # DENSE-AUL qp_info flags: the spill form ran; the literal multiplier update ran
N_CPU = 1000
BATCHES = {"default": dict(seed=5, tau_max=None), "tau25": dict(seed=6, tau_max=25.0)}


def near_limit(n, k=4, margin=0.02, speed=2.0, mode_mix=(0.34, 0.33, 0.33), pushes=True, terrain=False, seed=5, start=0):
    """Robots [start, start + n) of S.make's instance stream (same seed, modes, pushes and terrain) with k joints per robot
    moved to within `margin` rad of a limit (S.QMIN / S.QMAX, the controller's table) and moving towards it at up to `speed`
    rad/s.  The joints, the side and the distances come from the same block-keyed streams as S.make, so robot i is the same
    whatever the batch size or offset.  The desired CoM and swing-foot positions move with the robot's new kinematics."""
    sc = S.make(n, mode_mix=mode_mix, pushes=pushes, terrain=terrain, seed=seed, start=start)
    parts = []
    for blk in range(start // S.BLOCK, (start + n - 1) // S.BLOCK + 1):
        g = lambda s: S._rng(seed, blk, s)
        lo = max(start, blk * S.BLOCK) - blk * S.BLOCK
        hi = min(start + n, (blk + 1) * S.BLOCK) - blk * S.BLOCK
        joints = np.argsort(g(40).uniform(size=(12, S.BLOCK)), axis=0)[:k]
        upper = g(41).uniform(size=(k, S.BLOCK)) < 0.5
        dist = g(42).uniform(0.0, margin, (k, S.BLOCK))
        vel = g(43).uniform(0.0, speed, (k, S.BLOCK))
        parts.append([a[:, lo:hi] for a in (joints, upper, dist, vel)])
    joints, upper, dist, vel = (np.concatenate([p[i] for p in parts], axis=1) for i in range(4))
    cols = np.broadcast_to(np.arange(n), joints.shape)
    com0, feet0 = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["q"][joints, cols] = np.where(upper, S.QMAX[joints] - dist, S.QMIN[joints] + dist)
    sc["dq"][joints, cols] = np.where(upper, vel, -vel)
    com, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    sc["com_des_pos"][0:3] += (com - com0).T
    idx = np.arange(n)
    first = np.where(sc["mode"] == S.MODE_SWING_BL_FR, 1, 0)
    second = np.where(sc["mode"] == S.MODE_SWING_BL_FR, 3, 2)
    sc["sw_des_pos"] += np.hstack([feet[idx, first] - feet0[idx, first], feet[idx, second] - feet0[idx, second]]).T
    return sc


def row_families(nrows, neq):
    """Inequality-row indices (into L) of the torque-limit and joint-limit rows (wbc_oracle.c, the QP assembly)."""
    if neq == 18:                                      # stance: 20 friction rows, then 24 torque and 24 joint rows
        return np.arange(38, 62), np.arange(62, 86)
    return np.arange(22, 46), np.arange(58, 82)       # swing: 10 friction rows, 24 torque, 12 swing-tracking, 24 joint rows


def oracle_params(oracle, tau_max):
    p = oracle.default_params()
    if tau_max is not None:
        p.tau_max = tau_max
    return p


def build_batch(oracle, emu, dual, seed, tau_max, n=N_CPU):
    """Assemble the batch's QPs (observer wrench 0), decide feasibility with the LP, certify x* of each feasible QP and run
    the emulations: DENSE-AUL at reference settings (reduced and literal multiplier update) and at qp_epsx = 1e-4, exact mode."""
    sc = near_limit(n, seed=seed)
    qps = assemble(oracle, sc, range(n), w=np.zeros((n, 6)), params=oracle_params(oracle, tau_max))
    d = dict(qps=qps, sc=sc)
    d["t"] = np.array([P.lp_margin(L, neq)[0] for _, _, L, neq in qps])
    d["feas"] = d["t"] <= 0.0
    d["xd"], d["std"], d["infod"], _ = dual.solve_all(qps)
    for key, kw in (("ref", dict(kkt_mode=1)), ("lit", dict(kkt_mode=0)), ("tight", dict(epsx=1e-4))):
        r = [emu.qp_solve(Q, c, L, neq, **kw) for Q, c, L, neq in qps]
        d["x_" + key] = np.array([a[0] for a in r])
        d["ist_" + key] = np.array([a[1] for a in r])
    xs = np.zeros((n, 30))
    act_joint, act_torque, act_ineq, neqs = np.zeros(n, bool), np.zeros(n, bool), np.zeros(n, int), np.zeros(n, int)
    for k, (Q, c, L, neq) in enumerate(qps):
        if not d["feas"][k]:
            continue
        x, lam, W, _, _ = P.certified_qp(Q, c, L, neq, x0=d["xd"][k])
        xs[k] = x
        A, b = L[:, :30], L[:, 30]
        r = (A @ x - b) / np.maximum(1.0, np.maximum(np.abs(b), np.abs(A) @ np.abs(x)))
        on = np.zeros(L.shape[0], bool)
        on[neq:] = r[neq:] > -1e-9
        tq, jt = row_families(L.shape[0], neq)
        act_joint[k], act_torque[k], act_ineq[k], neqs[k] = on[jt].any(), on[tq].any(), on.sum(), neq
    d.update(xs=xs, act_joint=act_joint, act_torque=act_torque, act_ineq=act_ineq, over_kacap=(neqs + act_ineq > 36) & d["feas"])
    return d


@pytest.fixture(scope="module")
def dual():
    return DualEmu()


@pytest.fixture(scope="module")
def batches(oracle, emu, dual):
    return {name: build_batch(oracle, emu, dual, **kw) for name, kw in BATCHES.items()}


def errs(x, xs, idx):
    return np.array([E.err(x[k], xs[k]) for k in idx])


# ---------------------------------------------------------------------------------------------------------------------
# 1. the batches reach the regime, and the reference decides every instance

def coverage(d):
    f = d["feas"]
    ist = d["ist_ref"]
    return dict(n=len(f), infeasible=int((~f).sum()), joint=float(d["act_joint"][f].mean()), torque=float(d["act_torque"][f].mean()),
                over18=int((d["act_ineq"][f] > 18).sum()), over_kacap=int(d["over_kacap"].sum()), max_active=int(d["act_ineq"][f].max()),
                spill=int(((ist[:, 6] & SPILL) != 0).sum()), literal=int(((ist[:, 6] & LITERAL) != 0).sum()),
                max_work=int(ist[:, 4].max()))


# floors at about half of what was measured on 1 000 robots per batch (default / tau25): LP-infeasible 118 / 313, a joint-limit
# row active at x* on 97.5 / 97.7 % of the feasible QPs, a torque-limit row on 52.8 / 90.0 %, more than 18 active inequality
# rows on 4 / 14, DENSE-AUL instances that spill 517 / 731 and that take the literal multiplier update 582 / 779 (reference
# settings, reduced update), largest DENSE-AUL working set 67 / 67 inequality rows (MAXNIC = 72)
FLOORS = {"default": dict(infeasible=60, joint=0.8, torque=0.25, over18=2, spill=250, literal=290),
          "tau25": dict(infeasible=150, joint=0.8, torque=0.45, over18=7, spill=360, literal=390)}


@pytest.mark.parametrize("name", sorted(BATCHES))
def test_coverage_guard(batches, name):
    """The near-limit batches reach the regime they are for (FLOORS); a generator that drifts back inside the limits fails
    here (with margin = 1.0 rad: no infeasible QP, no spill).  Shares are over the LP-feasible QPs; an inequality row counts
    as active at x* when its row-scaled residual is above -1e-9.

    Not reached: an active set at x* larger than KACAP = 36 rows.  The most active inequality rows measured at an optimum is
    20 (on a swing QP, 12 equalities), and no optimum of either batch has more than 36 active rows.  The literal multiplier
    update still runs on more than half of the instances: there the reduced update declines on DENSE-AUL's working set, which
    is much larger than the optimum's active set (up to 67 rows), or on a dependent or ambiguous set."""
    c = coverage(batches[name])
    print("coverage %s: %s" % (name, c))
    for k, floor in FLOORS[name].items():
        assert c[k] >= floor, (name, k, c[k], floor)
    assert c["max_work"] > 18


def test_reference_lp_margin_and_restart(batches):
    """lp_margin on QPs with a known answer: a.x <= -1 and -a.x <= -1 cannot both hold, and the least row-scaled violation is
    exactly 1; a known-answer QP is feasible and the LP's point meets its inequality rows with slack -t*.  certified_qp refuses
    the infeasible QP.  On the near-limit QPs qp_exact.exact_qp stalls from a cold start on some instances (cycling, or a
    singular KKT matrix): certified_qp certifies those through the restart from the LP's point, with the x* it finds from the
    exact solver's x."""
    rng = np.random.default_rng(33)
    Q, c, L, xs, lam, act = E.known_answer_qp(rng, 20, 2, nact=3)
    t, xf = P.lp_margin(L, 2)
    r = (L[2:, :30] @ xf - L[2:, 30]) / np.maximum(1.0, np.abs(L[2:, 30]))
    assert t < 0 and r.max() <= t + 1e-9 and np.abs(L[:2, :30] @ xf - L[:2, 30]).max() <= 1e-9
    assert E.err(P.certified_qp(Q, c, L, 2)[0], xs) <= 1e-12
    a = rng.standard_normal(30)
    Lb = np.vstack([L, np.r_[a, -1.0], np.r_[-a, -1.0]])
    t, _ = P.lp_margin(Lb, 2)
    assert abs(t - 1.0) <= 1e-9
    with pytest.raises(E.CertificationError):
        P.certified_qp(Q, c, Lb, 2)
    d = batches["default"]
    stalled = []
    for k in np.flatnonzero(d["feas"]):
        Q, c, L, neq = d["qps"][k]
        x, _, _, _, how = P.certified_qp(Q, c, L, neq)
        if how == "lp restart":
            stalled.append(k)
        assert E.err(x, d["xs"][k]) <= 1e-12, k
    print("qp_exact.exact_qp failed from a cold start on %d of %d feasible QPs; all certified through the restart"
          % (len(stalled), d["feas"].sum()))
    assert stalled


def test_reference_decides_every_instance(batches):
    """Every QP is either LP-infeasible or has a certified x* (build_batch raises otherwise), and the LP's margin is far from
    zero on both sides, so the split does not depend on a tolerance."""
    for name, d in batches.items():
        t = d["t"]
        print("%s: %d infeasible of %d, smallest |t*| %.3e" % (name, int((t > 0).sum()), len(t), np.abs(t).min()))
        assert np.abs(t).min() >= 1e-4
        assert np.isfinite(t).all()


# ---------------------------------------------------------------------------------------------------------------------
# 2. the host emulations

def test_exact_mode_emulation(batches):
    """Exact mode: status 0 exactly on the LP-feasible QPs, within 1e-9 of x* there; WBC_ST_INFEASIBLE with x = 0 on the rest."""
    for name, d in batches.items():
        f = d["feas"]
        assert np.array_equal(d["std"] == 0, f), name
        assert (d["std"][~f] == ST_INFEASIBLE).all() and not d["xd"][~f].any(), name
        e = errs(d["xd"], d["xs"], np.flatnonzero(f))
        print("exact emulation %s: worst err %.3e over %d feasible QPs" % (name, e.max(), f.sum()))
        assert e.max() <= 1e-9


# DENSE-AUL on the feasible QPs, per (batch, setting): ceiling on the share that uses the rule's second branch, and the
# instances (index in the batch) allowed to meet neither branch.  Measured: default 0.475 / 0.494 / 0.471 with {508, 724, 959},
# {508, 959}, {508, 724, 959}; tau25 0.646 / 0.674 / 0.646 with none.
AUL_CEIL = {("default", "ref"): (0.55, {508, 724, 959}), ("default", "lit"): (0.55, {508, 959}),
            ("default", "tight"): (0.55, {508, 724, 959}),
            ("tau25", "ref"): (0.72, set()), ("tau25", "lit"): (0.72, set()), ("tau25", "tight"): (0.72, set())}


@pytest.mark.parametrize("name", sorted(BATCHES))
@pytest.mark.parametrize("key", ["ref", "lit", "tight"])
def test_dense_aul_emulation(batches, key, name):
    """DENSE-AUL at reference settings (reduced and literal multiplier update) and at qp_epsx = 1e-4 on the feasible QPs.

    The 0.5 % cap on the rule's second branch (qp_exact.MAX_SECOND) does not hold near the limits: about half of the
    instances (AUL_CEIL) stop with constraints violated by more than 1e-6.  qp_epsx = 1e-4 changes nothing here: these solves
    never meet even the 1e-2 feasibility test twice in a row, so both settings run all five outer iterations and stop on the
    iteration count, with the same x on every instance.

    Neither branch (pinned, AUL_CEIL): instance 508 of the default batch stops 13.0 from x* with a violation of 12.0 (err / v =
    1.09, just past K_VIOL = 1); 724 and 959 stop 2.2e-7 and 1.3e-7 from x* with violations of 3.5e-7 and 2.8e-7, below the
    1e-6 floor of the second branch.  Both are the augmented-Lagrangian iteration stopping on its count: the distance to x* of
    a point violating ill-conditioned active rows is not bounded by its violation.  Whether the reference ALGLIB stops at the
    same points is checked by test_neither_branch_cases_match_the_reference_alglib where the reference is built."""
    d = batches[name]
    f = np.flatnonzero(d["feas"])
    assert (d["ist_" + key][:, 0] == 2).all()
    T = E.Tally("DENSE-AUL %s %s" % (key, name))
    for k in f:
        T.add(int(k), E.err(d["x_" + key][k], d["xs"][k]), E.violation(d["x_" + key][k], d["qps"][k][2], d["qps"][k][3]))
    share = len(T.second) / T.n
    print(T.report() + ", second-branch share %.3f, neither: %s" % (share, [(i, "%.2e" % e, "%.2e" % v) for i, e, v in T.failed]))
    ceil_share, allowed = AUL_CEIL[(name, key)]
    assert share <= ceil_share, (name, key, share)
    assert {i for i, _, _ in T.failed} <= allowed, (name, key, T.failed)


def test_neither_branch_cases_match_the_reference_alglib(batches, oracle, have_ref):
    """The instances that meet neither branch, solved by the compiled reference ALGLIB at reference settings: the emulation
    (literal multiplier update, the reference's form) takes its decisions, i.e. the same Cholesky count and x within 1e-9."""
    d = batches["default"]
    for k in sorted(AUL_CEIL[("default", "ref")][1]):
        Q, c, L, neq = d["qps"][k]
        xr, nch, rc = oracle.ref_qp_solve(Q, c, L, neq)
        assert rc == 0
        print("instance %d: reference ALGLIB ncholesky %d, emulation %d, |x - x_emu| %.3e"
              % (k, nch, d["ist_lit"][k][1], E.err(xr, d["x_lit"][k])))
        assert nch == d["ist_lit"][k][1] and E.err(xr, d["x_lit"][k]) <= 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# 3. the CUDA kernels

def _opt_solve(batch, qps, **kw):
    """The OPT operator (wbc_qp_solve) on a list of QPs, one call per shape; returns x [n,30], status, info [n,8]."""
    n = len(qps)
    x, status, info = np.zeros((n, 30)), np.zeros(n, np.int32), np.zeros((n, 8), np.int32)
    for shape, ks in by_shape(qps).items():
        sub = [qps[k] for k in ks]
        r = batch.qp_solve(np.array([q[0] for q in sub]), np.array([q[1] for q in sub]),
                           np.array([q[2] for q in sub]).reshape(len(sub), shape[0], 31), shape[1], **kw)
        x[ks], status[ks], info[ks] = r[0], r[1], r[2]
    return x, status, info


# x distance to the emulation where the Cholesky counts agree.  Near the limits DENSE-AUL stops on its iteration count at a
# large penalty, and rounding is amplified: a host build of the emulation with FMA contraction (g++ -ffp-contract=fast
# -march=native) against the default one, on the two CPU batches, agrees on 98.0 / 98.7 % of the counts and differs there by
# up to 4.9e-5 / 8.1e-5 (1e-9 is exceeded on 323 / 507 instances).  Measured on a B200: 2.6e-5 / 9.6e-5 (OPT operator),
# 8.6e-5 (cycle).
TOL_X_SAME = 3e-4
# The spill and literal-update flags are decisions too, and rounding flips them on the odd instance: the FMA build of the
# emulation differs from the default one on 1 of the default batch's 1 000 instances in each flag (none in tau25), the first
# with equal Cholesky counts.  Measured on a B200: 2 of 1 000 in each flag of the default batch (instances 7 and 797 spill,
# 7 and 842 literal update: 797 and 842 are the FMA build's), none in tau25, none in the 4 096-robot cycle.  At most 1 % of
# the instances may differ.
MAX_FLAG_FLIPS = 0.01


def _flag_flips(what, got, want):
    flips = np.flatnonzero(got != want)
    print("%s: set on %d (emulation %d), differs on %d %s" % (what, got.sum(), want.sum(), len(flips), flips[:10].tolist()))
    assert got.sum() > 0 and len(flips) <= MAX_FLAG_FLIPS * len(got), what


def _rel(a, b):
    return np.abs(a - b).max(axis=1) / np.maximum(1.0, np.abs(b).max(axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BATCHES))
def test_gpu_opt_operator_default_mode(gpu_batch, batches, name):
    """Default mode takes the emulation's decisions on the near-limit QPs: Cholesky counts equal on >= 97 % (measured on a B200:
    97.5 / 99.0 %), x within TOL_X_SAME of the emulation's there (not the dense tests' 1e-9: see TOL_X_SAME), and the spill form
    (517 / 731 instances) and the literal multiplier update run where they run in the emulation, up to MAX_FLAG_FLIPS."""
    d = batches[name]
    x, status, info = _opt_solve(gpu_batch, d["qps"])
    assert (status == 0).all()
    same = info[:, 0] == d["ist_ref"][:, 1]
    rel = _rel(x, d["x_ref"])
    print("GPU OPT operator %s: ncholesky equal on %.4f, worst x distance there %.3e (elsewhere %.3e)"
          % (name, same.mean(), rel[same].max(), rel[~same].max() if (~same).any() else 0.0))
    assert same.mean() >= 0.97
    assert rel[same].max() <= TOL_X_SAME
    _flag_flips("GPU OPT operator %s spill" % name, (info[:, 5] & SPILL) != 0, (d["ist_ref"][:, 6] & SPILL) != 0)
    _flag_flips("GPU OPT operator %s literal update" % name, (info[:, 5] & LITERAL) != 0, (d["ist_ref"][:, 6] & LITERAL) != 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BATCHES))
def test_gpu_opt_operator_exact_and_warm(gpu_batch, batches, name):
    """Exact mode and its warm start give x* (within 1e-9) on the LP-feasible QPs and WBC_ST_INFEASIBLE with x = 0 on the
    rest: cold, then warm from the cold solve's own active sets, then warm from every row (each dropped as needed)."""
    d = batches[name]
    f = d["feas"]
    fi = np.flatnonzero(f)
    xc, stc, _ = _opt_solve(gpu_batch, d["qps"], exact=True)
    results = {"exact": (xc, stc)}
    n = len(d["qps"])
    for what in ("warm, cold sets", "warm, own sets", "warm, all rows"):
        xw, stw = np.zeros((n, 30)), np.zeros(n, np.int32)
        for shape, ks in by_shape(d["qps"]).items():
            sub = [d["qps"][k] for k in ks]
            Q, c, L = (np.array([q[i] for q in sub]) for i in range(3))
            act = None
            if what == "warm, own sets":
                act = gpu_batch.qp_solve(Q, c, L, shape[1], exact=True, warm=True)[4]
            elif what == "warm, all rows":
                act = np.full((len(ks), 3), 0xFFFFFFFF, np.uint32)
            r = gpu_batch.qp_solve(Q, c, L, shape[1], exact=True, warm=True, active=act)
            xw[ks], stw[ks] = r[0], r[1]
        results[what] = (xw, stw)
    for what, (x, st) in results.items():
        e = errs(x, d["xs"], fi)
        print("GPU %s %s: worst err %.3e over %d feasible, %d infeasible" % (what, name, e.max(), f.sum(), (~f).sum()))
        assert np.array_equal(st == 0, f), what
        assert (st[~f] == ST_INFEASIBLE).all() and not x[~f].any(), what
        assert e.max() <= 1e-9, what


N_CYCLE = 4096


@pytest.fixture(scope="module")
def cycle_scenario(emu):
    """4 096 near-limit robots (seed 7) and the emulation's cycle on them (default parameters, observer on)."""
    sc = near_limit(N_CYCLE, seed=7)
    return sc, emu.cycle(sc)


def _run_cycles(sc, express, fifo, ncycles=2):
    """`ncycles` cycles of the same inputs and observer state on a fresh ctx (the second one dispatches longest-first from
    the first one's costs, unless fifo)."""
    import os
    from wbc_quadruped_dob_b200 import api
    n = sc["mode"].shape[0]
    if express is not None:
        os.environ["WBC_EXPRESS"] = express
    try:
        b = api.WbcBatch(max_batch=n)
    finally:
        os.environ.pop("WBC_EXPRESS", None)
    b.fifo_dispatch = fifo
    try:
        outs = []
        for _ in range(ncycles):
            b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
            outs.append(b.cycle(sc))
        b.solver_shape()
        kernel = b.last_solver_kernel
    finally:
        b.close()
    return outs, kernel


@pytest.mark.gpu
def test_gpu_cycle_one_warp_per_solve(cycle_scenario):
    """The one-warp-per-solve kernel on 4 096 near-limit robots, with express lanes on and off (WBC_EXPRESS=0) and with FIFO
    and longest-first dispatch: against the emulation's cycle (status equal, Cholesky counts equal on >= 97 %, x within
    TOL_X_SAME where they are), the spill flag as in the emulation up to MAX_FLAG_FLIPS, and every variant bit-identical.  Measured on a B200:
    counts equal on 98.0 %, x within 8.6e-5 there, 2 128 of 4 096 instances spilled, working sets up to 69 rows."""
    sc, ref = cycle_scenario
    runs = {}
    for express in (None, "0"):
        for fifo in (False, True):
            outs, kernel = _run_cycles(sc, express, fifo)
            assert kernel == "wbc_solve_kernel"
            runs[(express, fifo)] = outs
    got = runs[(None, False)][1]
    assert np.array_equal(got["status"], ref["status"]) and (got["status"] == 0).all()
    same = got["qp_info"][0] == ref["qp_info"][0]
    rel = _rel(got["x"].T, ref["x"].T)
    print("GPU cycle (one warp per solve) %d near-limit robots: ncholesky equal on %.4f, worst x distance there %.3e, largest "
          "working set %d" % (N_CYCLE, same.mean(), rel[same].max(), got["qp_info"][3].max()))
    assert same.mean() >= 0.97 and rel[same].max() <= TOL_X_SAME
    _flag_flips("GPU cycle spill", (got["qp_info"][5] & SPILL) != 0, (ref["qp_info"][5] & SPILL) != 0)
    for key, outs in runs.items():
        for o, r in zip(outs, runs[(None, False)]):
            for k in ("tau", "w", "x", "qp_obj", "status"):
                assert np.array_equal(o[k], r[k]), (key, k)
            assert np.array_equal(o["qp_info"][:6], r["qp_info"][:6]), key


@pytest.mark.gpu
def test_gpu_cycle_stage_tasks_match_one_warp_per_solve():
    """The stage-task kernel (WBC_SOLVER=staged) against the one-warp-per-solve kernel (mono) on 49 152 near-limit robots, with
    the four-lane front kernel and with WBC_FRONT=thread: every output and every QP record bit for bit, spilled instances
    among them (measured on a B200: 26 655 of 49 152 with the four-lane front kernel, 26 657 with the thread one)."""
    import os
    from wbc_quadruped_dob_b200 import api
    n = 49152
    sc = near_limit(n, seed=9)
    for front in ("leg", "thread"):
        res = {}
        for solver in ("staged", "mono"):
            os.environ["WBC_SOLVER"], os.environ["WBC_FRONT"] = solver, front
            try:
                b = api.WbcBatch(max_batch=n)
            finally:
                del os.environ["WBC_SOLVER"], os.environ["WBC_FRONT"]
            try:
                b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
                o = b.cycle(sc)
                b.solver_shape()
                res[solver] = (o, b.qp_records(n), b.last_solver_kernel)
            finally:
                b.close()
        (o1, r1, k1), (o2, r2, k2) = res["staged"], res["mono"]
        assert (k1, k2) == ("wbc_solve_staged_kernel", "wbc_solve_kernel")
        spilled = [int(((o["qp_info"][5] & SPILL) != 0).sum()) for o in (o1, o2)]
        print("front %s: spilled instances, staged kernel %d, mono kernel %d of %d; failed %d" % (front, spilled[0], spilled[1], n,
                                                                                              int((o1["status"] != 0).sum())))
        assert spilled[0] > 0 and spilled[1] > 0
        for k in o1:
            assert np.array_equal(o1[k], o2[k]), (front, k)
        assert np.array_equal(r1, r2), front


def _exact_qp_fn(oracle, dual):
    """The oracle's QP solver for exact mode: x* where the LP finds the QP feasible, x = 0 where it does not."""
    def solve(Q, c, L, nrows, neq, x, nchol, term):
        Qa = np.ctypeslib.as_array(Q, (900,)).reshape(30, 30).copy()
        ca = np.ctypeslib.as_array(c, (30,)).copy()
        La = np.ctypeslib.as_array(L, (nrows * 31,)).reshape(nrows, 31).copy()
        xs = np.zeros(30)
        if P.lp_margin(La, neq)[0] <= 0.0:
            xs = P.certified_qp(Qa, ca, La, neq, x0=dual.solve(Qa, ca, La, neq)[0])[0]
        for k in range(30):
            x[k] = xs[k]
        if nchol:
            nchol[0] = 1
        if term:
            term[0] = 2
        return 0
    return oracle.QP_FN(solve)


@pytest.mark.gpu
def test_gpu_exact_cycle_infeasible_instances(oracle, dual):
    """Exact-mode cycle on 1 024 near-limit robots with tau_max = 25: WBC_ST_INFEASIBLE on exactly the LP-infeasible
    instances (the QPs assembled with the cycle's own w), x = 0 there and tau from x = 0 (the live oracle solving with x*, or
    x = 0 where the LP finds no point: tau within 1e-6 on every instance), x within 1e-9 of x* elsewhere; the observer state
    advances as in default mode (the estimate runs before the solve); the stored warm-start sets of the failed instances are
    cleared; with hold_tau_on_failure = 1 the failed instances get the last good torque."""
    from wbc_quadruped_dob_b200 import api
    n = 1024
    sc = near_limit(n, seed=8)
    inside = S.make(n, mode_mix=(0.34, 0.33, 0.33), pushes=True, seed=8)      # the same robots inside their limits
    p = api.default_params()
    p.tau_max = 25.0
    op = oracle_params(oracle, 25.0)
    b = api.WbcBatch(max_batch=n, params=p)
    try:
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        before = b.cycle(inside, exact=True)
        assert (before["status"] == 0).all() and b.get_active_set(n)[3].all()
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        got = b.cycle(sc, exact=True)
        obs_exact, sets = b.get_observer_state(n), b.get_active_set(n)
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        b.cycle(sc)
        obs_default = b.get_observer_state(n)
        p.hold_tau_on_failure = 1
        b.set_params(p)
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        b.cycle(inside, exact=True)
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        held = b.cycle(sc, exact=True)
    finally:
        b.close()
    qps = assemble(oracle, sc, range(n), w=[got["w"][:, i] for i in range(n)], params=op)
    feas = np.array([P.lp_margin(L, neq)[0] <= 0.0 for _, _, L, neq in qps])
    bad = ~feas
    print("exact cycle, tau_max 25: %d of %d LP-infeasible, status -22 on %d" % (bad.sum(), n, (got["status"] == ST_INFEASIBLE).sum()))
    assert bad.sum() > 0
    assert np.array_equal(got["status"] == ST_INFEASIBLE, bad) and (got["status"][feas] == 0).all()
    assert not got["x"][:, bad].any()
    e = np.array([E.err(got["x"][:, k], P.certified_qp(Q, c, L, neq, x0=got["x"][:, k])[0]) for k, (Q, c, L, neq) in enumerate(qps) if feas[k]])
    print("exact cycle: worst err %.3e over %d feasible" % (e.max(), feas.sum()))
    assert e.max() <= 1e-9
    ref, _ = oracle.run_cycle_batch(sc, params=op, nthreads=1, solver=_exact_qp_fn(oracle, dual))
    et = util.rel_rows(got["tau"].T, ref["tau"])
    print("exact cycle vs live oracle (x* or x = 0): worst tau rel err %.3e, on the infeasible instances %.3e" % (et.max(), et[bad].max()))
    assert et.max() <= 1e-6
    for a, bb in zip(obs_exact, obs_default):
        assert np.array_equal(a, bb)
    assert not sets[:, bad].any() and sets[3, feas].all()
    assert np.array_equal(held["status"], got["status"])
    assert np.array_equal(held["tau"][:, bad], before["tau"][:, bad])
    assert np.array_equal(held["tau"][:, feas], got["tau"][:, feas])
