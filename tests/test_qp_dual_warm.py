"""Warm start of the exact-mode QP solver (csrc/qp_dual.cuh, solve_dual with WARM = true; wbc_qp_solve_warm, WBC_QP_WARM).

A warm set is only a guess: whatever it holds, the result must be the optimum x* certified by tests/qp_exact.py (err <= 1e-9, as
for the cold solver in test_qp_dual.py), and the status must be the cold status.  Every QP set of test_qp_dual.py is started from
  (a) its own cold final active set,        (b) random subsets of its inequality rows,      (c) every inequality row,
  (d) the complement of (a),                (e) the final set of a perturbed neighbour QP,  (f) (a) with bits set at the
                                                                                                equality rows and beyond nrows.
With (a) the GI loop should add no row at all; across the cases it adds far fewer rows than a cold solve.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import qp_exact as E
from tests import util
from tests.test_qp_dual import DualEmu, controller_qps, dual, worst_err  # noqa: F401  (module fixtures)
from tests.test_qp_exact import SHAPES, by_shape, known_answer_batch

_dp = C.POINTER(C.c_double)
_up = C.POINTER(C.c_uint)
TOL = 1e-9
ST_INFEASIBLE, ST_NOT_PD = -22, -23
CASES = "abcdef"


class WarmEmu(DualEmu):
    """DualEmu (the cold solve) plus the g++ build of the warm start, tests/host_emu/qp_dual_warm_emu.cpp (test infrastructure only)."""

    def __init__(self):
        super().__init__()
        so = os.path.join(util.EMU_DIR, "libqp_dual_warm_emu.so")
        util._build_emu(os.path.join(util.EMU_DIR, "qp_dual_warm_emu.cpp"), so)
        self.wlib = C.CDLL(so)
        self.wlib.emu_qp_dual_solve_warm.argtypes = [_dp, _dp, _dp, C.c_int, C.c_int, _dp, C.POINTER(C.c_int), _dp, _up]

    def solve_warm(self, Q, c, L, neq, mask):
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        c = np.ascontiguousarray(c, dtype=np.float64)
        L = np.ascontiguousarray(L, dtype=np.float64).reshape(-1, 31)
        x = np.zeros(30)
        info = (C.c_int * 8)()
        fl = C.c_double()
        act = (C.c_uint * 3)(*[int(v) for v in mask])
        st = self.wlib.emu_qp_dual_solve_warm(Q.ctypes.data_as(_dp), c.ctypes.data_as(_dp), L.ctypes.data_as(_dp), L.shape[0], int(neq),
                                             x.ctypes.data_as(_dp), info, C.byref(fl), act)
        return x, int(st), list(info), fl.value, np.array(list(act), dtype=np.uint32)


@pytest.fixture(scope="module")
def warm():
    return WarmEmu()


def to_mask(rows):
    m = np.zeros(3, dtype=np.uint32)
    for r in rows:
        m[r >> 5] |= np.uint32(1 << (r & 31))
    return m


def from_mask(m):
    return [r for r in range(96) if (int(m[r >> 5]) >> (r & 31)) & 1]


def gi_adds(info):
    """inequality rows the GI loop added: all additions less the warm ones and the equalities (never dropped)"""
    return info[1] - info[6] - (info[4] - info[3])


def warm_sets(warm, Q, c, L, neq, cold_mask, rng):
    """the warm sets (a)..(f) of one QP"""
    nrows = L.shape[0]
    ineq = list(range(neq, nrows))
    a = cold_mask
    b = to_mask([r for r in ineq if rng.uniform() < 0.3])
    cc = to_mask(ineq)
    d = to_mask([r for r in ineq if r not in set(from_mask(a))])
    # (e): a neighbour QP -- c and the right-hand sides moved by a few per cent of their scale
    c2 = c + 0.02 * np.abs(c).max() * rng.standard_normal(30)
    L2 = L.copy()
    if nrows:
        L2[:, 30] += 0.02 * np.maximum(1.0, np.abs(L[:, 30])) * rng.standard_normal(nrows)
    e = warm.solve_warm(Q, c2, L2, neq, np.zeros(3, np.uint32))[4]
    f = a | to_mask(list(range(neq)) + list(range(nrows, 96)))
    return dict(a=a, b=b, c=cc, d=d, e=e, f=f)


def run_cases(warm, qps, xs, seed, what):
    """solve every QP cold and from each warm set; check err, status and masks; return the per-case GI additions"""
    rng = np.random.default_rng(seed)
    cold_gi, gi = [], {k: [] for k in CASES}
    worst = 0.0
    for (Q, c, L, neq), x_star in zip(qps, xs):
        L = np.asarray(L).reshape(-1, 31)
        x0, st0, info0, _, m0 = warm.solve_warm(Q, c, L, neq, np.zeros(3, np.uint32))
        cold_gi.append(gi_adds(info0))
        for k, m in warm_sets(warm, Q, c, L, neq, m0, rng).items():
            x, st, info, _, mout = warm.solve_warm(Q, c, L, neq, m)
            assert st == st0, (what, k, st, st0)
            if st != 0:
                assert not x.any() and not mout.any()
                continue
            e = E.err(x, x_star)
            worst = max(worst, e)
            assert e <= TOL, (what, k, e, info)
            assert from_mask(mout) == [r for r in from_mask(mout) if neq <= r < L.shape[0]]
            assert bin(int(mout[0])).count("1") + bin(int(mout[1])).count("1") + bin(int(mout[2])).count("1") == info[3]
            gi[k].append(gi_adds(info))
    return np.array(cold_gi), {k: np.array(v) for k, v in gi.items()}, worst


def report(what, cold_gi, gi, worst):
    print("%s: worst err %.3e; GI additions cold %.2f, warm %s; (a) without a GI addition on %.4f"
          % (what, worst, cold_gi.mean(), " ".join("%s %.2f" % (k, v.mean()) for k, v in gi.items() if len(v)),
             np.mean(gi["a"] == 0) if len(gi["a"]) else 1.0))


# ---------------------------------------------------------------------------------------------------------------------
# 1. the host emulation

def test_all_zero_warm_set_is_the_cold_solve(warm, controller_qps):
    for Q, c, L, neq in controller_qps["qps"][:256]:
        xw, stw, infow, flw, _ = warm.solve_warm(Q, c, L, neq, np.zeros(3, np.uint32))
        x, st, info, fl = warm.solve(Q, c, L, neq)
        assert stw == st and np.array_equal(xw, x) and infow[:6] == info[:6] and infow[6:] == [0, 0] and flw == fl


@pytest.mark.parametrize("shape", SHAPES + [(20, 0), (60, 30)])
def test_warm_known_answers(warm, shape):
    qps, xs = known_answer_batch(shape, 2000, 48)
    cold_gi, gi, w = run_cases(warm, qps, xs, 7 + shape[0], "known answers %s" % (shape,))
    report("warm emulation %s" % (shape,), cold_gi, gi, w)
    assert np.mean(gi["a"] == 0) >= 0.99


def test_warm_controller_qps(warm, controller_qps):
    d = controller_qps
    cold_gi, gi, w = run_cases(warm, d["qps"], d["xs"], 11, "controller QPs")
    report("warm emulation, 4096 controller QPs", cold_gi, gi, w)
    assert np.mean(gi["a"] == 0) >= 0.99
    every = np.concatenate(list(gi.values()))
    assert every.mean() <= 0.5 * cold_gi.mean()
    assert gi["e"].mean() <= 0.25 * cold_gi.mean()


def test_warm_golden_qps(warm):
    for name in ("qp_stance", "qp_swing"):
        z = np.load(util.GOLDEN + "/" + name + ".npz")
        neq = int(z["neq"])
        qps = [(z["Q"][k], z["c"][k], z["L"][k], neq) for k in range(z["Q"].shape[0])]
        xs = [E.exact_qp(Q, c, L, neq, x0=warm.solve(Q, c, L, neq)[0])[0] for Q, c, L, _ in qps]
        cold_gi, gi, w = run_cases(warm, qps, xs, 13, name)
        report("warm emulation, golden " + name, cold_gi, gi, w)
        assert np.mean(gi["a"] == 0) >= 0.99


def test_warm_degenerate_vertices_and_dependent_equalities(warm):
    rng = np.random.default_rng(31)
    qps, xs = [], []
    for _ in range(24):
        Q, c, L, x_star, lam, act = E.known_answer_qp(rng, 40, 5, nact=8)
        ina = [i for i in act if i >= 5]
        extra = []
        for _ in range(6):
            w = rng.uniform(0.0, 1.0, len(ina))
            w[rng.integers(0, len(ina))] = 0.0
            extra.append(w @ L[ina])
        qps.append((Q, c, np.vstack([L, np.array(extra)]), 5))
        xs.append(x_star)
    rng = np.random.default_rng(32)
    Q, c, L, x_star, _, _ = E.known_answer_qp(rng, 40, 6, nact=5)
    qps.append((Q, c, np.vstack([L[:6], 2.0 * L[2:3], L[6:]]), 7))
    xs.append(x_star)
    cold_gi, gi, w = run_cases(warm, qps, xs, 17, "degenerate")
    report("warm emulation, degenerate vertices", cold_gi, gi, w)


def test_warm_failures_keep_their_status(warm):
    rng = np.random.default_rng(33)
    Q, c, L, _, _, _ = E.known_answer_qp(rng, 20, 2, nact=3)
    a = rng.standard_normal(30)
    Lb = np.vstack([L, np.r_[a, -1.0], np.r_[-a, -1.0]])
    bad = np.vstack([L[:2], L[1:2] * 2.0 + np.r_[np.zeros(30), 1.0], L[2:]])
    Hn = np.diag(np.r_[np.ones(29), -1.0])
    for QQ, LL, neq, want in ((Q, Lb, 2, ST_INFEASIBLE), (Q, bad, 3, ST_INFEASIBLE), (Hn, L, 2, ST_NOT_PD)):
        nrows = LL.shape[0]
        for m in (to_mask(range(neq, nrows)), to_mask([nrows - 1, nrows - 2]), to_mask(range(96))):
            x, st, info, _, mout = warm.solve_warm(QQ, c, LL, neq, m)
            assert st == want and not x.any() and not mout.any()


def test_warm_no_rows_and_all_rows(warm):
    rng = np.random.default_rng(35)
    Q, c, _, x_star, _, _ = E.known_answer_qp(rng, 0, 0)
    for m in (np.zeros(3, np.uint32), to_mask(range(96))):
        x, st, info, _, mout = warm.solve_warm(Q, c, np.zeros((0, 31)), 0, m)
        assert st == 0 and E.err(x, x_star) <= TOL and info[1] == 0 and info[6] == 0 and not mout.any()
    qps, xs = [], []
    for _ in range(12):
        Q, c, L, x_star, _, act = E.known_answer_qp(rng, 86, 18)
        qps.append((Q, c, L, 18))
        xs.append(x_star)
    cold_gi, gi, w = run_cases(warm, qps, xs, 19, "86 rows")
    report("warm emulation, 86 rows", cold_gi, gi, w)
    assert (gi["a"] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# 2. the CUDA kernel (wbc_qp_solve_warm)

@pytest.mark.gpu
def test_gpu_dense_warm_matches_the_emulation(gpu_batch, warm, controller_qps):
    d = controller_qps
    rng = np.random.default_rng(23)
    worst_emu = worst_star = 0.0
    for shape, ks in by_shape(d["qps"]).items():
        sub = [d["qps"][k] for k in ks]
        n = len(sub)
        Q, c = np.array([q[0] for q in sub]), np.array([q[1] for q in sub])
        L = np.array([q[2] for q in sub]).reshape(n, shape[0], 31)
        x0, st0, info0, _, m0 = gpu_batch.qp_solve(Q, c, L, shape[1], exact=True, warm=True, active=np.zeros((n, 3), np.uint32))
        assert (st0 == 0).all() and (info0[:, 6] == 0).all()
        sets = [warm_sets(warm, Q[j], c[j], L[j], shape[1], m0[j], rng) for j in range(n)]
        for k in CASES:
            m = np.array([s[k] for s in sets], dtype=np.uint32)
            x, st, info, _, mout = gpu_batch.qp_solve(Q, c, L, shape[1], exact=True, warm=True, active=m.copy())
            assert (st == 0).all()
            for j in range(n):
                xe, ste, infoe, _, me = warm.solve_warm(Q[j], c[j], L[j], shape[1], m[j])
                de = np.abs(x[j] - xe).max() / max(1.0, np.abs(xe).max())
                worst_emu = max(worst_emu, de)
                worst_star = max(worst_star, E.err(x[j], d["xs"][ks[j]]))
                assert de <= 1e-10 and E.err(x[j], d["xs"][ks[j]]) <= TOL, (shape, k, j)
                # the mask round-trips: it is the final active set, and solving from it again needs no GI addition
                assert bin(int(mout[j][0])).count("1") + bin(int(mout[j][1])).count("1") + bin(int(mout[j][2])).count("1") == info[j][3]
            x2, st2, info2, _, m2 = gpu_batch.qp_solve(Q, c, L, shape[1], exact=True, warm=True, active=mout.copy())
            assert (st2 == 0).all() and np.mean(info2[:, 1] - info2[:, 6] - (info2[:, 4] - info2[:, 3]) == 0) >= 0.99
            assert np.abs(x2 - x).max() <= 1e-9 * max(1.0, np.abs(x).max())
    print("GPU wbc_qp_solve_warm, 4096 controller QPs x 6 warm sets: worst distance to the emulation %.3e, worst err %.3e"
          % (worst_emu, worst_star))


@pytest.mark.gpu
def test_gpu_dense_warm_failures_and_refusals(gpu_batch):
    from wbc_quadruped_dob_b200 import api
    rng = np.random.default_rng(33)
    Q, c, L, _, _, _ = E.known_answer_qp(rng, 20, 2, nact=3)
    a = rng.standard_normal(30)
    Lb = np.vstack([L, np.r_[a, -1.0], np.r_[-a, -1.0]])
    full = np.tile(to_mask(range(96)), (1, 1))
    x, st, _, _, m = gpu_batch.qp_solve(Q[None], c[None], Lb[None], 2, exact=True, warm=True, active=full.copy())
    assert st[0] == ST_INFEASIBLE and not x.any() and not m.any()
    Hn = np.diag(np.r_[np.ones(29), -1.0])
    x, st, _, _, m = gpu_batch.qp_solve(Hn[None], c[None], L[None], 2, exact=True, warm=True, active=full.copy())
    assert st[0] == ST_NOT_PD and not x.any() and not m.any()
    Qnan = Q.copy(); Qnan[3, 1] = np.nan
    x, st, _, _, m = gpu_batch.qp_solve(Qnan[None], c[None], L[None], 2, exact=True, warm=True, active=full.copy())
    assert st[0] == -21 and not x.any() and not m.any()
    with pytest.raises(api.WbcError):
        gpu_batch.qp_solve(Q[None], c[None], L[None], 2, warm=True, active=full.copy())
    act = np.full((1, 3), 7, np.uint32)
    xs = np.full((1, 30), 7.25)
    rc = gpu_batch.lib.wbc_qp_solve_warm(gpu_batch.h, 1, Q.ctypes.data, c.ctypes.data, L.ctypes.data, 87, 2, xs.ctypes.data, None, None,
                                         None, act.ctypes.data, None, api.HOST_PTRS)
    assert rc != 0 and (xs == 7.25).all() and (act == 7).all()
    rc = gpu_batch.lib.wbc_qp_solve_warm(gpu_batch.h, 1, Q.ctypes.data, c.ctypes.data, L.ctypes.data, 20, 2, xs.ctypes.data, None, None,
                                         None, None, None, api.HOST_PTRS)
    assert rc != 0 and (xs == 7.25).all()


@pytest.mark.gpu
def test_gpu_dense_warm_device_pointer_path(gpu_batch, controller_qps):
    import torch
    from wbc_quadruped_dob_b200 import api
    qps = [q for q in controller_qps["qps"] if q[3] == 18][:300]
    Q = np.array([q[0] for q in qps]); c = np.array([q[1] for q in qps]); L = np.array([q[2] for q in qps])
    n, nrows = len(qps), L.shape[1]
    m0 = gpu_batch.qp_solve(Q, c, L, 18, exact=True, warm=True, active=np.zeros((n, 3), np.uint32))[4]
    host = gpu_batch.qp_solve(Q, c, L, 18, exact=True, warm=True, active=m0.copy())
    dQ, dc, dL = (torch.from_numpy(a).cuda() for a in (Q, c, L))
    dm = torch.from_numpy(m0.view(np.int32).copy()).cuda()
    dx = torch.full((n, 30), 7.25, dtype=torch.float64, device="cuda")
    dst = torch.full((n,), 5, dtype=torch.int32, device="cuda")
    dinfo = torch.zeros((n, 8), dtype=torch.int32, device="cuda")
    dfl = torch.zeros(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    api._check(gpu_batch.lib.wbc_qp_solve_warm(gpu_batch.h, n, dQ.data_ptr(), dc.data_ptr(), dL.data_ptr(), nrows, 18, dx.data_ptr(),
                                               dst.data_ptr(), dinfo.data_ptr(), dfl.data_ptr(), dm.data_ptr(),
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream), api.DEVICE_PTRS), "wbc_qp_solve_warm")
    for got, want in zip((dx, dst, dinfo, dfl), host[:4]):
        assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(dm.cpu().numpy().view(np.uint32), host[4])


# ---------------------------------------------------------------------------------------------------------------------
# 3. the C++ host layer: wbc_b200::OPT with warm_start

SRC = os.path.join(util.ROOT, "tests", "cpp", "opt_warm_host.cpp")
EXE = os.path.join(util.ROOT, "tests", "cpp", "opt_warm_host.bin")


@pytest.mark.gpu
def test_cpp_opt_warm_golden_qps(tmp_path):
    """Each golden QP twice through one OPT with exact_qp and warm_start: the second pass starts from the first pass's set."""
    from wbc_quadruped_dob_b200 import build as B
    lib = B.build()
    libdir = os.path.dirname(lib)
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(util.ROOT, "include"), SRC, "-o", EXE,
                    "-L" + libdir, "-lwbc_b200", "-Wl,-rpath," + libdir], check=True)
    for name in ("qp_stance", "qp_swing"):
        z = np.load(util.GOLDEN + "/" + name + ".npz")
        neq, m = int(z["neq"]), z["Q"].shape[0]
        nrows = z["L"].shape[1]
        fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
        with open(fin, "wb") as f:
            np.array([m, nrows, neq], dtype=np.int32).tofile(f)
            for k in range(m):
                np.concatenate([z["Q"][k].ravel(), z["c"][k].ravel(), z["L"][k].ravel()]).astype(np.float64).tofile(f)
        subprocess.run([EXE, fin, fout], check=True)
        out = np.fromfile(fout, dtype=np.float64).reshape(2, m, 32)
        assert (out[:, :, 30] == 0).all()
        assert (out[1, :, 31] > 0).mean() >= 0.5        # the second pass was warm-started (rows forced in)
        for p in range(2):
            for k in range(m):
                xs = E.exact_qp(z["Q"][k], z["c"][k], z["L"][k], neq, x0=out[p, k, :30])[0]
                assert E.err(out[p, k, :30], xs) <= TOL, (name, p, k)
