"""The DENSE-AUL solver (csrc/qp_warp.cuh) against the exact optimum x* of each QP, certified by its KKT conditions
(tests/qp_exact.py), a reference that shares no code with the solver, its host emulation or the reference ALGLIB.

The live oracle's QP solver is the solver's own source built for the host wherever the reference ALGLIB is not built, so
the "vs live oracle" tests cannot see a wrong working-set decision, multiplier update or stopping test written into
qp_warp.cuh.  These tests can.

Tolerance rule (qp_exact.passes), with err = max|x - x*| / max(1, max|x*|) and v(x) the solver's largest row-scaled
constraint violation: err <= 1e-7, or v(x) > 1e-6 and err <= 1 * v(x), the second branch for at most 0.5 % of a group.
At the reference settings DENSE-AUL may stop on its epsx = 1e-2 criterion with constraints still violated, and then lands
that far from x*; raising qp_outerits does not change that, a tighter qp_epsx does.  With qp_epsx = 1e-4 the rule is a
flat err <= 1e-7.

Calibration on the host emulation (g++ -ffp-contract=off), 2 x 2 048 assembled controller QPs (seeds 100 and 101, 40 %
stance, pushes, terrain on / off, observer wrench [0.3, -0.2, 0.5, 0.01, -0.02, 0.03]): reduced and literal multiplier
updates alike, 2 instances use the second branch (worst err 1.3e-5, err/v 0.079), all others within 1e-8 of x*; at
qp_epsx = 1e-4 the worst err is 6.1e-9.  The known-answer QPs of SHAPES (96 per shape) are within 2.4e-8 of x* at qp_epsx = 1e-4.

On a B200 (sm_100a, FMA contraction on) the same 4 096 QPs give the emulation's numbers: the same 2 second-branch
instances, worst err 1.2e-8 at qp_epsx = 1e-4, Cholesky counts equal to the emulation's on 99.8 % (reduced update) and
99.6 % (literal).  Cycle solutions: standing_4096 within 1.7e-8 of x*; the terrain/push mixes and trot_65536 use the second
branch on 2 of 3 000, 4 of 4 096 and 4 of 1 500 instances (worst err/v 0.5).
"""
import ctypes as C

import numpy as np
import pytest

from tests import qp_exact as E
from tests import util
from wbc_quadruped_dob_b200 import scenarios as S

W_OBS = [0.3, -0.2, 0.5, 0.01, -0.02, 0.03]      # the observer wrench of tests/golden/qp_*.npz
SHAPES = [(0, 0), (1, 0), (1, 1), (12, 12), (30, 30), (40, 5), (72, 0), (86, 14), (86, 18)]


def assemble(oracle, sc, idx, w=None, params=None):
    """The controller's dense QPs (oracle.assemble_only): list of (Q, c, L, neq)."""
    out = []
    for k, i in enumerate(idx):
        _, qp = oracle.assemble_only(sc, int(i), params=params, w=W_OBS if w is None else w[k])
        out.append((np.array(qp.Q).reshape(30, 30), np.array(qp.c), np.array(qp.L)[:qp.nrows * 31].reshape(qp.nrows, 31), qp.neq))
    return out


def exact_all(qps, x0s):
    """x* and f* of every QP, warm-started from a solver's x."""
    xs = np.array([E.exact_qp(Q, c, L, neq, x0=x0)[0] for (Q, c, L, neq), x0 in zip(qps, x0s)])
    fs = np.array([E.objective(Q, c, x) for (Q, c, _, _), x in zip(qps, xs)])
    return xs, fs


def tally(what, qps, x, xs, flat=False):
    """The rule over a group; instances are numbered by their position in qps."""
    T = E.Tally(what, flat=flat)
    for k, ((_, _, L, neq), xk, xsk) in enumerate(zip(qps, x, xs)):
        T.add(k, E.err(xk, xsk), E.violation(xk, L, neq))
    return T


def check_objective(what, T, obj, fs):
    """The objective matches f* to 1e-9 relative wherever x met the first branch of the rule."""
    second = {i for i, _, _ in T.second}
    keep = np.array([k not in second for k in range(len(fs))])
    rel = np.abs(obj - fs)[keep] / np.maximum(1.0, np.abs(fs[keep]))
    print("%s: worst objective rel err %.3e" % (what, rel.max() if rel.size else 0.0))
    assert rel.max() <= 1e-9, what


def by_shape(qps):
    """Group the QPs by (nrows, neq) (stance and swing): {shape: list of indices}."""
    g = {}
    for k, (_, _, L, neq) in enumerate(qps):
        g.setdefault((L.shape[0], neq), []).append(k)
    return g


def emu_solve_all(emu, qps, **kw):
    res = [emu.qp_solve(Q, c, L, neq, **kw) for Q, c, L, neq in qps]
    return np.array([r[0] for r in res]), np.array([r[1][0] for r in res]), np.array([r[1][1] for r in res])


# ---------------------------------------------------------------------------------------------------------------------
# 1. the reference itself

@pytest.mark.parametrize("shape", SHAPES + [(20, 0), (60, 30)])
def test_reference_recovers_known_answers(shape):
    nrows, neq = shape
    rng = np.random.default_rng(1000 + 100 * nrows + neq)
    for _ in range(12):
        Q, c, L, xs, lam, act = E.known_answer_qp(rng, nrows, neq)
        for x0 in (None, xs + 0.3 * rng.standard_normal(30)):
            x, l, W, cert = E.exact_qp(Q, c, L, neq, x0=x0)
            assert E.err(x, xs) <= 1e-12, cert
            assert W == act
            assert nrows == 0 or np.abs(l - lam).max() <= 1e-9 * max(1.0, np.abs(lam).max())


def test_reference_refuses_what_it_cannot_certify():
    rng = np.random.default_rng(7)
    Q, c, L, xs, lam, act = E.known_answer_qp(rng, 40, 5, nact=6)
    A, b, H = L[:, :30], L[:, 30], E.sym_lower(Q)
    E.certify(H, c, A, b, 5, xs, lam)
    with pytest.raises(E.CertificationError):                   # not stationary
        E.certify(H, c, A, b, 5, xs + 1e-6, lam)
    bad = lam.copy(); bad[act[-1]] = -bad[act[-1]]               # wrong sign of an inequality multiplier
    with pytest.raises(E.CertificationError):
        E.certify(H, c + 2 * A[act[-1]] * lam[act[-1]], A, b, 5, xs, bad)
    off = [i for i in range(5, 40) if i not in act][0]           # a multiplier on a slack row
    bad = lam.copy(); bad[off] = 1.0
    with pytest.raises(E.CertificationError):
        E.certify(H, c - A[off], A, b, 5, xs, bad)
    bb = b.copy(); bb[act[-1]] -= 1e-3                           # infeasible
    with pytest.raises(E.CertificationError):
        E.certify(H, c, A, bb, 5, xs, lam)
    Hn = H.copy(); Hn[0, 0] = -1.0                               # not strictly convex: no unique optimum
    with pytest.raises(E.CertificationError):
        E.exact_qp(Hn, c, L, 5)


def test_reference_reproduces_golden_alglib_solutions():
    """The reference ALGLIB's stored x of the 32 golden QPs is within 3.4e-9 of x* (measured: 2.0e-9 stance, 3.4e-9 swing)."""
    for name in ("qp_stance", "qp_swing"):
        z = np.load(util.GOLDEN + "/" + name + ".npz")
        for k in range(z["Q"].shape[0]):
            x, _, _, _ = E.exact_qp(z["Q"][k], z["c"][k], z["L"][k], int(z["neq"]), x0=z["x"][k])
            assert E.err(z["x"][k], x) <= 3.4e-9, (name, k)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the tolerance rule on the host emulation

@pytest.fixture(scope="module")
def controller_qps(oracle, emu):
    """4 096 assembled controller QPs (40 % stance, pushes; terrain on for seed 100, off for seed 101), the emulation's x
    at reference settings with both multiplier updates and at qp_epsx = 1e-4, and x*, f* of each."""
    qps = []
    for seed, terrain in ((100, True), (101, False)):
        sc = S.make(2048, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=terrain, seed=seed)
        qps += assemble(oracle, sc, range(2048))
    d = dict(qps=qps)
    d["emu1"], d["st1"], d["nch1"] = emu_solve_all(emu, qps, kkt_mode=1)
    d["emu0"], d["st0"], d["nch0"] = emu_solve_all(emu, qps, kkt_mode=0)
    d["emu4"], d["st4"], _ = emu_solve_all(emu, qps, epsx=1e-4)
    d["xs"], d["fs"] = exact_all(qps, d["emu1"])
    return d


@pytest.mark.parametrize("kkt_mode", [1, 0])
def test_emulation_meets_the_rule_on_controller_qps(controller_qps, kkt_mode):
    d = controller_qps
    assert (d["st%d" % kkt_mode] == 2).all()
    x = d["emu%d" % kkt_mode]
    T = tally("emulation kkt_mode %d" % kkt_mode, d["qps"], x, d["xs"])
    T.check()
    check_objective("emulation kkt_mode %d" % kkt_mode, T, np.array([E.objective(Q, c, xk) for (Q, c, _, _), xk in zip(d["qps"], x)]), d["fs"])


def test_emulation_tight_stop_is_exact(controller_qps):
    d = controller_qps
    assert (d["st4"] == 2).all()
    tally("emulation qp_epsx 1e-4", d["qps"], d["emu4"], d["xs"], flat=True).check()


def test_emulation_two_multiplier_updates_agree(controller_qps):
    d = controller_qps
    diff = np.array([E.err(a, b) for a, b in zip(d["emu0"], d["emu1"])])
    print("emulation literal vs reduced update: worst %.3e, p99 %.3e, ncholesky equal %.4f"
          % (diff.max(), np.percentile(diff, 99), np.mean(d["nch0"] == d["nch1"])))
    assert diff.max() <= 1e-8 and np.percentile(diff, 99) <= 1e-9       # measured: 1.8e-9, 2.7e-11


def known_answer_batch(shape, seed, n):
    nrows, neq = shape
    rng = np.random.default_rng(seed + 100 * nrows + neq)
    qa = [E.known_answer_qp(rng, nrows, neq) for _ in range(n)]
    return [(q[0], q[1], q[2], neq) for q in qa], [q[3] for q in qa]


@pytest.mark.parametrize("shape", SHAPES)
def test_emulation_meets_the_rule_on_known_answers(emu, shape):
    """Random well-conditioned QPs need the tight stop: at reference settings 1 of 864 (86 rows, 14 equalities) stopped
    9.3e-6 from x* with a violation of only 2.7e-7."""
    qps, xs = known_answer_batch(shape, 2000, 48)
    x, st, _ = emu_solve_all(emu, qps, epsx=1e-4)
    assert (st == 2).all()
    tally("emulation qp_epsx 1e-4 %s" % (shape,), qps, x, xs, flat=True).check()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the CUDA kernels

def _gpu_solve(batch, qps, idx=None):
    """Solve the QPs through the OPT operator, one call per (nrows, neq); returns x [n,30], status, info [n,8], flops."""
    n = len(qps)
    x, status, info, flops = np.zeros((n, 30)), np.zeros(n, np.int32), np.zeros((n, 8), np.int32), np.zeros(n)
    for shape, ks in by_shape(qps).items():
        sub = [qps[k] for k in ks]
        r = batch.qp_solve(np.array([q[0] for q in sub]), np.array([q[1] for q in sub]),
                           np.array([q[2] for q in sub]).reshape(len(sub), shape[0], 31), shape[1])
        x[ks], status[ks], info[ks], flops[ks] = r
    return x, status, info, flops


def _with_params(batch, **kw):
    from wbc_quadruped_dob_b200 import api
    p = api.default_params()
    for k, v in kw.items():
        setattr(p, k, v)
    batch.set_params(p)


def _restore(batch):
    from wbc_quadruped_dob_b200 import api
    batch.set_params(api.default_params())


@pytest.mark.gpu
def test_opt_operator_controller_qps(gpu_batch, controller_qps):
    d = controller_qps
    x, status, info, _ = _gpu_solve(gpu_batch, d["qps"])
    assert (status == 0).all()
    T = tally("GPU OPT operator", d["qps"], x, d["xs"])
    T.check()
    check_objective("GPU OPT operator", T, np.array([E.objective(Q, c, xk) for (Q, c, _, _), xk in zip(d["qps"], x)]), d["fs"])
    agree = np.mean(info[:, 0] == d["nch1"])
    print("GPU OPT operator: ncholesky equal to the emulation's on %.4f" % agree)
    assert agree >= 0.97


@pytest.mark.gpu
def test_opt_operator_literal_multiplier_update(gpu_batch, controller_qps):
    d = controller_qps
    x_red, _, _, _ = _gpu_solve(gpu_batch, d["qps"])
    _with_params(gpu_batch, qp_literal_kkt=1)
    try:
        x, status, info, _ = _gpu_solve(gpu_batch, d["qps"])
    finally:
        _restore(gpu_batch)
    assert (status == 0).all()
    tally("GPU literal KKT update", d["qps"], x, d["xs"]).check()
    agree = np.mean(info[:, 0] == d["nch0"])
    print("GPU literal KKT update: ncholesky equal to the emulation's on %.4f" % agree)
    assert agree >= 0.97
    diff = np.array([E.err(a, b) for a, b in zip(x, x_red)])
    emu_diff = np.array([E.err(a, b) for a, b in zip(d["emu0"], d["emu1"])])
    print("literal vs reduced update: GPU worst %.3e p99 %.3e; emulation worst %.3e p99 %.3e"
          % (diff.max(), np.percentile(diff, 99), emu_diff.max(), np.percentile(emu_diff, 99)))
    assert diff.max() <= max(4 * emu_diff.max(), 1e-8)
    assert np.percentile(diff, 99) <= max(4 * np.percentile(emu_diff, 99), 1e-9)


@pytest.mark.gpu
def test_opt_operator_tight_stop(gpu_batch, controller_qps):
    d = controller_qps
    _with_params(gpu_batch, qp_epsx=1e-4)
    try:
        x, status, _, _ = _gpu_solve(gpu_batch, d["qps"])
    finally:
        _restore(gpu_batch)
    assert (status == 0).all()
    tally("GPU qp_epsx 1e-4", d["qps"], x, d["xs"], flat=True).check()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
def test_opt_operator_shapes(gpu_batch, emu, shape):
    """Known-answer QPs at the OPT operator's extreme and controller shapes: the GPU takes the emulation's decisions at
    reference settings and at qp_epsx = 1e-4, and with the tight stop lands within 1e-7 of x*.  The Cholesky counts are
    pooled over the two settings: FMA contraction alone flips a count on 2-3 % of these random QPs (a g++ -ffp-contract=fast
    build of the emulation against the default one: 0.969 at (1, 1) and (72, 0) for one setting, x still within 4e-11)."""
    nrows, neq = shape
    qps, xs = known_answer_batch(shape, 3000, 96)
    n = len(qps)
    Q, c, L = np.array([q[0] for q in qps]), np.array([q[1] for q in qps]), np.array([q[2] for q in qps]).reshape(n, nrows, 31)
    same_all = []
    for epsx in (1e-2, 1e-4):
        _with_params(gpu_batch, qp_epsx=epsx)
        try:
            x, status, info, _ = gpu_batch.qp_solve(Q, c, L, neq)
        finally:
            _restore(gpu_batch)
        xe, ste, nche = emu_solve_all(emu, qps, epsx=epsx)
        assert np.array_equal(status == 0, ste == 2) and (status == 0).all()
        same = info[:, 0] == nche
        same_all.append(same)
        rel = np.abs(x - xe).max(axis=1) / np.maximum(1.0, np.abs(xe).max(axis=1))
        print("GPU shape %s qp_epsx %g: ncholesky equal to the emulation's on %.4f, worst x distance there %.3e, elsewhere %.3e"
              % (shape, epsx, same.mean(), rel[same].max(), rel[~same].max() if (~same).any() else 0.0))
        assert rel[same].max() <= 1e-9
    assert np.concatenate(same_all).mean() >= 0.97
    tally("GPU qp_epsx 1e-4 %s" % (shape,), qps, x, xs, flat=True).check()


def _raw_qp_solve(batch, n, nrows, neq, Q=None, c=None, L=None):
    """wbc_qp_solve with explicit counts and sentinel-filled outputs; returns the outputs (raises WbcError on refusal)."""
    from wbc_quadruped_dob_b200 import api
    m = max(n, 1)
    Q = np.zeros((m, 30, 30)) if Q is None else Q
    c = np.zeros((m, 30)) if c is None else c
    L = np.zeros((m, max(nrows, 1), 31)) if L is None else L
    out = dict(x=np.full((m, 30), 7.25), status=np.full(m, 5, np.int32), info=np.full((m, 8), 5, np.int32), flops=np.full(m, 7.25))
    api._check(batch.lib.wbc_qp_solve(batch.h, n, Q.ctypes.data, c.ctypes.data, L.ctypes.data, nrows, neq, out["x"].ctypes.data,
                                      out["status"].ctypes.data, out["info"].ctypes.data, out["flops"].ctypes.data, None, api.HOST_PTRS),
               "wbc_qp_solve")
    return out


@pytest.mark.gpu
def test_opt_operator_refuses_bad_shapes_without_side_effects(gpu_batch):
    from wbc_quadruped_dob_b200 import api
    z = np.load(util.GOLDEN + "/qp_stance.npz")
    before = gpu_batch.qp_solve(z["Q"], z["c"], z["L"], int(z["neq"]))
    shape_before = gpu_batch.solver_shape()
    for nrows, neq in ((87, 12), (73, 0), (10, 11), (-1, 0), (5, -1), (0, -1)):
        with pytest.raises(api.WbcError):
            _raw_qp_solve(gpu_batch, 4, nrows, neq, L=np.zeros((4, 87, 31)))
    with pytest.raises(api.WbcError):
        _raw_qp_solve(gpu_batch, -1, 86, 18)
    small = api.WbcBatch(max_batch=8, device=0)
    try:
        with pytest.raises(api.WbcError):
            _raw_qp_solve(small, 9, 86, 18)
        out = _raw_qp_solve(small, 8, 86, 18, Q=np.ascontiguousarray(z["Q"][:8]), c=np.ascontiguousarray(z["c"][:8]),
                            L=np.ascontiguousarray(z["L"][:8]))
        assert np.array_equal(out["x"], before[0][:8])
    finally:
        small.close()
    after = gpu_batch.qp_solve(z["Q"], z["c"], z["L"], int(z["neq"]))
    for a, b in zip(before, after):
        assert np.array_equal(a, b)
    assert gpu_batch.solver_shape() == shape_before


@pytest.mark.gpu
def test_refused_call_leaves_outputs_untouched(gpu_batch):
    from wbc_quadruped_dob_b200 import api
    m = 4
    x = np.full((m, 30), 7.25)
    st = np.full(m, 5, np.int32)
    Q, c, L = np.zeros((m, 30, 30)), np.zeros((m, 30)), np.zeros((m, 87, 31))
    rc = gpu_batch.lib.wbc_qp_solve(gpu_batch.h, m, Q.ctypes.data, c.ctypes.data, L.ctypes.data, 87, 12, x.ctypes.data, st.ctypes.data,
                                    None, None, None, api.HOST_PTRS)
    assert rc != 0
    assert (x == 7.25).all() and (st == 5).all()


def _mixed_pool(oracle, n):
    sc = S.make(n, mode_mix=(1.0, 0.0, 0.0), pushes=True, terrain=True, seed=444)
    return assemble(oracle, sc, range(n))


@pytest.mark.gpu
def test_grid_and_tail_solve_every_instance_once(oracle):
    """The dense kernel's grid is min(n, resident solver CTAs): batch sizes around it and past several rounds of the work
    queue give, for every instance, bit for bit what the same QP gives solved alone; reversing the batch reverses the outputs."""
    import torch
    from wbc_quadruped_dob_b200 import api
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    pool = _mixed_pool(oracle, 61)
    Q = np.array([q[0] for q in pool]); c = np.array([q[1] for q in pool]); L = np.array([q[2] for q in pool]); neq = pool[0][3]
    b = api.WbcBatch(max_batch=8192, device=0)
    try:
        ctas, _, g = b.solver_shape()
        print("solver grid %d = %d CTAs x %d SMs" % (g, ctas, sm))
        assert g == ctas * sm
        alone = [b.qp_solve(Q[k:k + 1], c[k:k + 1], L[k:k + 1], neq) for k in range(len(pool))]
        for n in (1, 31, 33, g - 1, g, g + 1, 3 * g + 7):
            assert n <= 8192
            sel = (np.arange(n) * 7 + n) % len(pool)        # the instance -> QP map changes with n: a skipped instance shows
            x, status, info, flops = b.qp_solve(Q[sel], c[sel], L[sel], neq)
            for k in range(len(pool)):
                m = sel == k
                if not m.any():
                    continue
                ax, ast, ainf, afl = alone[k]
                assert (x[m] == ax).all() and (status[m] == ast).all() and (info[m] == ainf).all() and (flops[m] == afl).all(), (n, k)
            r = b.qp_solve(Q[sel[::-1]], c[sel[::-1]], L[sel[::-1]], neq)
            for got, want in zip(r, (x, status, info, flops)):
                assert np.array_equal(got[::-1], want), n
    finally:
        b.close()


@pytest.mark.gpu
def test_only_the_lower_triangle_of_q_is_read(gpu_batch, emu, oracle):
    rng = np.random.default_rng(55)
    pool = _mixed_pool(oracle, 64)
    Q = np.array([q[0] for q in pool]); c = np.array([q[1] for q in pool]); L = np.array([q[2] for q in pool]); neq = pool[0][3]
    junk = Q + np.triu(rng.uniform(-1e3, 1e3, Q.shape), 1)
    a = gpu_batch.qp_solve(Q, c, L, neq)
    b = gpu_batch.qp_solve(junk, c, L, neq)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    for k in range(0, 64, 8):                       # the emulation reads the same triangle
        assert np.array_equal(emu.qp_solve(junk[k], c[k], L[k], neq)[0], emu.qp_solve(Q[k], c[k], L[k], neq)[0])
    qa = [E.known_answer_qp(rng, 40, 5) for _ in range(32)]
    Qk = np.array([q[0] for q in qa]); ck = np.array([q[1] for q in qa]); Lk = np.array([q[2] for q in qa])
    a = gpu_batch.qp_solve(Qk, ck, Lk, 5)
    b = gpu_batch.qp_solve(Qk + np.triu(rng.uniform(-1e3, 1e3, Qk.shape), 1), ck, Lk, 5)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.gpu
def test_device_pointer_path_equals_host_path(gpu_batch, oracle):
    import torch
    from wbc_quadruped_dob_b200 import api
    pool = _mixed_pool(oracle, 200)
    Q = np.array([q[0] for q in pool]); c = np.array([q[1] for q in pool]); L = np.array([q[2] for q in pool]); neq = pool[0][3]
    n, nrows = len(pool), L.shape[1]
    host = gpu_batch.qp_solve(Q, c, L, neq)
    dQ, dc, dL = (torch.from_numpy(a).cuda() for a in (Q, c, L))
    dx = torch.full((n, 30), 7.25, dtype=torch.float64, device="cuda")
    dst = torch.full((n,), 5, dtype=torch.int32, device="cuda")
    dinfo = torch.zeros((n, 8), dtype=torch.int32, device="cuda")
    dfl = torch.zeros(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    api._check(gpu_batch.lib.wbc_qp_solve(gpu_batch.h, n, dQ.data_ptr(), dc.data_ptr(), dL.data_ptr(), nrows, neq, dx.data_ptr(), dst.data_ptr(),
                                          dinfo.data_ptr(), dfl.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream),
                                          api.DEVICE_PTRS), "wbc_qp_solve")
    for got, want in zip((dx, dst, dinfo, dfl), host):
        assert np.array_equal(got.cpu().numpy(), want)


def _cycle_check(what, oracle, batch, sc, idx, params=None, oracle_params=None):
    """Run the cycle on the GPU, assemble the QP of each instance in idx with the GPU's w and apply the rule to the cycle's
    x and qp_obj."""
    if params is not None:
        batch.set_params(params)
    try:
        batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        got = batch.cycle(sc)
    finally:
        if params is not None:
            _restore(batch)
    assert (got["status"] == 0).all()
    qps = assemble(oracle, sc, idx, w=[got["w"][:, i] for i in idx], params=oracle_params)
    x = got["x"][:, idx].T
    xs, fs = exact_all(qps, x)
    T = tally(what, qps, x, xs)
    T.check()
    check_objective(what, T, got["qp_obj"][idx], fs)
    return got


@pytest.mark.gpu
def test_cycle_solutions_standing_4096(gpu_batch, oracle):
    sc = S.make_config("standing_4096")
    _cycle_check("cycle standing_4096", oracle, gpu_batch, sc, np.arange(4096))


@pytest.mark.gpu
def test_cycle_solutions_mixed_terrain_pushes(gpu_batch, oracle):
    sc = S.make(3000, mode_mix=(0.4, 0.3, 0.3), terrain=True, pushes=True, seed=12)
    _cycle_check("cycle mixed terrain pushes", oracle, gpu_batch, sc, np.arange(3000))


@pytest.mark.gpu
def test_cycle_solutions_65536_staged(gpu_batch, oracle):
    sc = S.make_config("trot_65536")
    _cycle_check("cycle trot_65536 (every 16th)", oracle, gpu_batch, sc, np.arange(0, 65536, 16))
    _, _, _ = gpu_batch.solver_shape()
    assert gpu_batch.last_solver_kernel == "wbc_solve_staged_kernel"


@pytest.mark.gpu
def test_cycle_solutions_fix_swing_rhs(gpu_batch, oracle, oracle_qp):
    """fix_swing_rhs = 1 (the swing rows' right-hand sides the reference leaves at zero): the cycle's QP solutions against x*
    of the QPs the oracle assembles with the same setting, and the cycle's torques against the oracle's."""
    from wbc_quadruped_dob_b200 import api
    sc = S.make(1500, mode_mix=(0.2, 0.4, 0.4), pushes=True, terrain=True, seed=13)
    p = api.default_params()
    p.fix_swing_rhs = 1
    op = oracle.default_params()
    op.fix_swing_rhs = 1
    got = _cycle_check("cycle fix_swing_rhs", oracle, gpu_batch, sc, np.arange(1500), params=p, oracle_params=op)
    ref, _ = oracle.run_cycle_batch(sc, params=op, nthreads=8, solver=oracle_qp)
    util.check_cycle_parity(got, ref, what="fix_swing_rhs")
