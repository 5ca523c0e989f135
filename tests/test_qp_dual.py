"""The exact-mode QP solver (csrc/qp_dual.cuh, WBC_QP_EXACT) against the certified KKT optimum x* of tests/qp_exact.py,
which shares no code with it.

Unlike DENSE-AUL at the reference's settings (tests/test_qp_exact.py), the exact solver stops at the optimum, so there is no
violation branch: err = max|x - x*| / max(1, max|x*|) <= 1e-9 on every instance.

Calibration on the host emulation (g++ -ffp-contract=off, tests/host_emu/qp_dual_emu.cpp):
  * known-answer QPs, 48 per shape of SHAPES and (20, 0), (60, 30): worst err 5.3e-13 (at (30, 30));
  * 4 096 assembled controller QPs (seeds 100 and 101, as in test_qp_exact.py): worst err 2.6e-14; rows added 18..31 (equalities
    included); drops 0/1/2/3/4/5 on 3329/622/124/17/3/1 instances; 0.14..0.26 MFLOP per solve;
  * the 32 golden QPs: worst err 1.9e-14.
On a B200 (FMA contraction on) the GPU meets the same bound on every instance, within 1e-10 of the emulation (measured with the
Givens-chain row addition: 2.6e-14, equal active inequality counts on 100 %).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import qp_exact as E
from tests import util
from tests.test_qp_exact import SHAPES, assemble, by_shape, known_answer_batch
from wbc_quadruped_dob_b200 import scenarios as S

_dp = C.POINTER(C.c_double)
TOL = 1e-9
ST_INFEASIBLE, ST_NOT_PD = -22, -23


class DualEmu:
    """g++ build of qp_dual.cuh with the single-lane executor (test infrastructure only)."""

    def __init__(self):
        so = os.path.join(util.EMU_DIR, "libqp_dual_emu.so")
        util._build_emu(os.path.join(util.EMU_DIR, "qp_dual_emu.cpp"), so)
        self.lib = C.CDLL(so)
        self.lib.emu_qp_dual_solve.argtypes = [_dp, _dp, _dp, C.c_int, C.c_int, _dp, C.POINTER(C.c_int), _dp]

    def solve(self, Q, c, L, neq):
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        c = np.ascontiguousarray(c, dtype=np.float64)
        L = np.ascontiguousarray(L, dtype=np.float64).reshape(-1, 31)
        x = np.zeros(30)
        info = (C.c_int * 8)()
        fl = C.c_double()
        st = self.lib.emu_qp_dual_solve(Q.ctypes.data_as(_dp), c.ctypes.data_as(_dp), L.ctypes.data_as(_dp), L.shape[0], int(neq),
                                        x.ctypes.data_as(_dp), info, C.byref(fl))
        return x, int(st), list(info), fl.value

    def solve_all(self, qps):
        r = [self.solve(Q, c, L, neq) for Q, c, L, neq in qps]
        return (np.array([a[0] for a in r]), np.array([a[1] for a in r]), np.array([a[2] for a in r]), np.array([a[3] for a in r]))


@pytest.fixture(scope="module")
def dual():
    return DualEmu()


def worst_err(x, xs):
    return max((E.err(a, b) for a, b in zip(x, xs)), default=0.0)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the host emulation

@pytest.mark.parametrize("shape", SHAPES + [(20, 0), (60, 30)])
def test_emulation_known_answers(dual, shape):
    qps, xs = known_answer_batch(shape, 2000, 48)
    x, st, info, _ = dual.solve_all(qps)
    assert (st == 0).all()
    assert (info[:, 0] == 1).all() and (info[:, 5] & 256).all()
    w = worst_err(x, xs)
    print("exact emulation %s: worst err %.3e" % (shape, w))
    assert w <= TOL


@pytest.fixture(scope="module")
def controller_qps(oracle, dual):
    """4 096 assembled controller QPs (as test_qp_exact.controller_qps), the emulation's x and x* of each."""
    qps = []
    for seed, terrain in ((100, True), (101, False)):
        sc = S.make(2048, mode_mix=(0.4, 0.3, 0.3), pushes=True, terrain=terrain, seed=seed)
        qps += assemble(oracle, sc, range(2048))
    x, st, info, flops = dual.solve_all(qps)
    xs = np.array([E.exact_qp(Q, c, L, neq, x0=x0)[0] for (Q, c, L, neq), x0 in zip(qps, x)])
    return dict(qps=qps, x=x, st=st, info=info, flops=flops, xs=xs)


def test_emulation_controller_qps(controller_qps):
    d = controller_qps
    assert (d["st"] == 0).all()
    e = np.array([E.err(a, b) for a, b in zip(d["x"], d["xs"])])
    adds, drops = d["info"][:, 1], d["info"][:, 2]
    print("exact emulation, 4096 controller QPs: worst err %.3e; additions %d..%d, drops histogram %s, flops %.0f..%.0f"
          % (e.max(), adds.min(), adds.max(), np.bincount(drops).tolist(), d["flops"].min(), d["flops"].max()))
    assert e.max() <= TOL
    for k, (_, _, L, neq) in enumerate(d["qps"]):
        assert E.violation(d["x"][k], L, neq) <= 1e-10


def test_emulation_golden_qps(dual):
    for name in ("qp_stance", "qp_swing"):
        z = np.load(util.GOLDEN + "/" + name + ".npz")
        neq = int(z["neq"])
        for k in range(z["Q"].shape[0]):
            x, st, _, _ = dual.solve(z["Q"][k], z["c"][k], z["L"][k], neq)
            assert st == 0
            xs = E.exact_qp(z["Q"][k], z["c"][k], z["L"][k], neq, x0=x)[0]
            assert E.err(x, xs) <= TOL, (name, k)


def test_emulation_degenerate_vertices(dual):
    """Extra rows through x* that are non-negative combinations of active rows (a degenerate vertex, like the 5 friction rows of
    an unloaded foot): the optimum is unchanged and the solver never adds a dependent row."""
    rng = np.random.default_rng(31)
    for _ in range(24):
        Q, c, L, xs, lam, act = E.known_answer_qp(rng, 40, 5, nact=8)
        ina = [i for i in act if i >= 5]
        extra = []
        for _ in range(6):
            w = rng.uniform(0.0, 1.0, len(ina))
            w[rng.integers(0, len(ina))] = 0.0
            extra.append(w @ L[ina])
        L2 = np.vstack([L, np.array(extra)])
        for LL in (L2, np.vstack([L2[:5], L2[5:][rng.permutation(L2.shape[0] - 5)]])):
            x, st, info, _ = dual.solve(Q, c, LL, 5)
            assert st == 0 and E.err(x, xs) <= TOL, (st, info, E.err(x, xs))
            assert info[4] <= 30


def test_emulation_dependent_equalities(dual):
    rng = np.random.default_rng(32)
    Q, c, L, xs, lam, act = E.known_answer_qp(rng, 40, 6, nact=5)
    dup = np.vstack([L[:6], 2.0 * L[2:3], L[6:]])                # a consistent duplicate (scaled) of equality 2
    x, st, info, _ = dual.solve(Q, c, dup, 7)
    assert st == 0 and E.err(x, xs) <= TOL
    assert info[5] & 512
    bad = dup.copy()
    bad[6, 30] += 1.0                                          # the same normal, another right-hand side
    x, st, _, _ = dual.solve(Q, c, bad, 7)
    assert st == ST_INFEASIBLE and not x.any()


def test_emulation_infeasible(dual):
    rng = np.random.default_rng(33)
    Q, c, L, xs, lam, act = E.known_answer_qp(rng, 20, 2, nact=3)
    a = rng.standard_normal(30)
    Lb = np.vstack([L, np.r_[a, -1.0], np.r_[-a, -1.0]])       # a.x <= -1 and a.x >= 1
    x, st, info, _ = dual.solve(Q, c, Lb, 2)
    assert st == ST_INFEASIBLE and not x.any()


def test_emulation_not_positive_definite(dual):
    rng = np.random.default_rng(34)
    Q, c, L, xs, lam, act = E.known_answer_qp(rng, 20, 2)
    U, _ = np.linalg.qr(rng.standard_normal((30, 30)))
    ev = np.linspace(1.0, 3.0, 30)
    ev[7] = -0.5                                               # indefinite, with a positive diagonal
    Hn = (U * ev) @ U.T
    assert (np.diag(Hn) > 0).any()
    for H in (Hn, np.diag(np.r_[np.ones(29), -1.0]), np.zeros((30, 30))):
        x, st, _, _ = dual.solve(H, c, L, 2)
        assert st == ST_NOT_PD and not x.any()


def test_emulation_no_rows_and_all_rows(dual):
    rng = np.random.default_rng(35)
    Q, c, L, xs, _, _ = E.known_answer_qp(rng, 0, 0)
    x, st, info, _ = dual.solve(Q, c, np.zeros((0, 31)), 0)
    assert st == 0 and E.err(x, xs) <= TOL and info[1] == 0 and info[4] == 0
    for _ in range(12):
        Q, c, L, xs, _, act = E.known_answer_qp(rng, 86, 18)
        x, st, info, _ = dual.solve(Q, c, L, 18)
        assert st == 0 and E.err(x, xs) <= TOL
        assert info[4] == len(act) and info[3] == len(act) - 18


# ---------------------------------------------------------------------------------------------------------------------
# 2. the CUDA kernel (wbc_qp_solve with WBC_QP_EXACT)

def _gpu_solve(batch, qps):
    n = len(qps)
    x, status, info, flops = np.zeros((n, 30)), np.zeros(n, np.int32), np.zeros((n, 8), np.int32), np.zeros(n)
    for shape, ks in by_shape(qps).items():
        sub = [qps[k] for k in ks]
        r = batch.qp_solve(np.array([q[0] for q in sub]), np.array([q[1] for q in sub]),
                           np.array([q[2] for q in sub]).reshape(len(sub), shape[0], 31), shape[1], exact=True)
        x[ks], status[ks], info[ks], flops[ks] = r
    return x, status, info, flops


@pytest.mark.gpu
def test_gpu_controller_qps(gpu_batch, controller_qps):
    d = controller_qps
    x, status, info, flops = _gpu_solve(gpu_batch, d["qps"])
    assert (status == 0).all()
    e = np.array([E.err(a, b) for a, b in zip(x, d["xs"])])
    dx = np.abs(x - d["x"]).max(axis=1) / np.maximum(1.0, np.abs(d["x"]).max(axis=1))
    same = np.mean(info[:, 3] == d["info"][:, 3])
    print("GPU exact, 4096 controller QPs: worst err %.3e, worst distance to the emulation %.3e, active inequality rows equal on %.4f"
          % (e.max(), dx.max(), same))
    assert e.max() <= TOL and dx.max() <= 1e-10 and same >= 0.995
    assert (info[:, 5] & 256).all() and (info[:, 0] == 1).all() and (flops > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES + [(20, 0), (60, 30)])
def test_gpu_known_answers(gpu_batch, dual, shape):
    nrows, neq = shape
    qps, xs = known_answer_batch(shape, 3000, 96)
    n = len(qps)
    Q, c, L = np.array([q[0] for q in qps]), np.array([q[1] for q in qps]), np.array([q[2] for q in qps]).reshape(n, nrows, 31)
    x, status, info, _ = gpu_batch.qp_solve(Q, c, L, neq, exact=True)
    xe, ste, infoe, _ = dual.solve_all(qps)
    assert (status == 0).all() and (ste == 0).all()
    dx = np.abs(x - xe).max(axis=1) / np.maximum(1.0, np.abs(xe).max(axis=1))
    print("GPU exact %s: worst err %.3e, distance to the emulation %.3e" % (shape, worst_err(x, xs), dx.max()))
    assert worst_err(x, xs) <= TOL and dx.max() <= 1e-10
    assert np.mean(info[:, 3] == infoe[:, 3]) >= 0.995


@pytest.mark.gpu
def test_gpu_golden_qps_and_edge_cases(gpu_batch, dual):
    for name in ("qp_stance", "qp_swing"):
        z = np.load(util.GOLDEN + "/" + name + ".npz")
        neq = int(z["neq"])
        x, status, _, _ = gpu_batch.qp_solve(z["Q"], z["c"], z["L"], neq, exact=True)
        assert (status == 0).all()
        for k in range(z["Q"].shape[0]):
            xs = E.exact_qp(z["Q"][k], z["c"][k], z["L"][k], neq, x0=x[k])[0]
            assert E.err(x[k], xs) <= TOL
    rng = np.random.default_rng(33)
    Q, c, L, _, _, _ = E.known_answer_qp(rng, 20, 2, nact=3)
    a = rng.standard_normal(30)
    Lb = np.vstack([L, np.r_[a, -1.0], np.r_[-a, -1.0]])
    x, status, _, _ = gpu_batch.qp_solve(Q[None], c[None], Lb[None], 2, exact=True)
    assert status[0] == ST_INFEASIBLE and not x.any()
    Hn = np.diag(np.r_[np.ones(29), -1.0])
    x, status, _, _ = gpu_batch.qp_solve(Hn[None], c[None], L[None], 2, exact=True)
    assert status[0] == ST_NOT_PD and not x.any()
    Qnan = Q.copy(); Qnan[3, 1] = np.nan
    x, status, _, _ = gpu_batch.qp_solve(Qnan[None], c[None], L[None], 2, exact=True)
    assert status[0] == -21 and not x.any()


@pytest.mark.gpu
def test_gpu_refuses_bad_shapes(gpu_batch):
    from wbc_quadruped_dob_b200 import api
    for nrows, neq in ((87, 12), (73, 0), (10, 11), (-1, 0), (5, -1)):
        x = np.full((4, 30), 7.25)
        Q, c, L = np.zeros((4, 30, 30)), np.zeros((4, 30)), np.zeros((4, 87, 31))
        rc = gpu_batch.lib.wbc_qp_solve(gpu_batch.h, 4, Q.ctypes.data, c.ctypes.data, L.ctypes.data, nrows, neq, x.ctypes.data, None,
                                        None, None, None, api.HOST_PTRS | api.QP_EXACT)
        assert rc != 0 and (x == 7.25).all()


@pytest.mark.gpu
def test_gpu_device_pointer_path(gpu_batch, controller_qps):
    import torch
    from wbc_quadruped_dob_b200 import api
    qps = [q for q in controller_qps["qps"] if q[3] == 18][:300]
    Q = np.array([q[0] for q in qps]); c = np.array([q[1] for q in qps]); L = np.array([q[2] for q in qps])
    n, nrows = len(qps), L.shape[1]
    host = gpu_batch.qp_solve(Q, c, L, 18, exact=True)
    dQ, dc, dL = (torch.from_numpy(a).cuda() for a in (Q, c, L))
    dx = torch.full((n, 30), 7.25, dtype=torch.float64, device="cuda")
    dst = torch.full((n,), 5, dtype=torch.int32, device="cuda")
    dinfo = torch.zeros((n, 8), dtype=torch.int32, device="cuda")
    dfl = torch.zeros(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    api._check(gpu_batch.lib.wbc_qp_solve(gpu_batch.h, n, dQ.data_ptr(), dc.data_ptr(), dL.data_ptr(), nrows, 18, dx.data_ptr(), dst.data_ptr(),
                                          dinfo.data_ptr(), dfl.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream),
                                          api.DEVICE_PTRS | api.QP_EXACT), "wbc_qp_solve")
    for got, want in zip((dx, dst, dinfo, dfl), host):
        assert np.array_equal(got.cpu().numpy(), want)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the C++ host layer: wbc_b200::OPT with exact_qp

SRC = os.path.join(util.ROOT, "tests", "cpp", "opt_exact_host.cpp")
EXE = os.path.join(util.ROOT, "tests", "cpp", "opt_exact_host.bin")


@pytest.mark.gpu
def test_cpp_opt_exact_golden_qps(tmp_path):
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
        out = np.fromfile(fout, dtype=np.float64).reshape(m, 31)
        assert (out[:, 30] == 0).all()
        for k in range(m):
            xs = E.exact_qp(z["Q"][k], z["c"][k], z["L"][k], neq, x0=out[k, :30])[0]
            assert E.err(out[k, :30], xs) <= TOL, (name, k)
