"""Host logic of the DEVICE code, compiled by g++ with the single-lane executor (tests/host_emu): the same headers the
CUDA kernels are built from, checked against the oracle and the golden fixtures without a GPU."""
import numpy as np
import pytest

from tests import util
from wbc_quadruped_dob_b200 import scenarios as S


@pytest.mark.parametrize("name", ["cycle_standing", "cycle_trot_pushes", "cycle_mixed_terrain"])
def test_device_code_matches_golden_cycle(emu, name):
    sc, gold = util.load_golden(name)
    got = emu.cycle(sc)
    util.check_cycle_parity(got, gold, what=name)
    assert np.abs(got["yd"].T - gold["yd"]).max() <= util.TOL_OBS
    assert np.abs(got["yw"].T - gold["yw"]).max() <= util.TOL_OBS
    assert np.abs(got["x"].T - gold["x"]).max() <= 1e-7 * max(1.0, np.abs(gold["x"]).max())
    # same discrete decisions as the reference solver: Cholesky counts (rep.ncholesky, opt.cpp:41325) agree except
    # where a last-bit difference flips one comparison (SURVEY.md Appendix F, ~1 in 2000) -- outputs still match
    assert np.mean(got["qp_info"][0] == gold["ncholesky"]) >= 0.97


def test_device_code_trot_replay_with_chained_observer(emu):
    sc, gold = util.load_golden("cycle_trot_replay")
    n = sc["mode"].shape[0]
    yd, yw = np.zeros((6, 1)), np.zeros((6, 1))
    for i in range(n):
        one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
        one["obs_yd"], one["obs_yw"] = yd, yw
        got = emu.cycle(one)
        yd, yw = got["yd"], got["yw"]
        assert np.abs(got["w"][:, 0] - gold["w"][i]).max() <= util.TOL_OBS * max(1.0, np.abs(gold["w"][i]).max())
        assert util.rel_rows(got["tau"].T, gold["tau"][i:i + 1]).max() <= util.TOL_TAU


@pytest.mark.parametrize("name", ["qp_stance", "qp_swing"])
def test_solver_restatement_matches_reference_alglib_golden(emu, name):
    z = np.load(util.GOLDEN + "/" + name + ".npz")
    for k in range(z["Q"].shape[0]):
        x, ist, flops = emu.qp_solve(z["Q"][k], z["c"][k], z["L"][k], int(z["neq"]))
        assert ist[0] == 2
        assert ist[1] == z["ncholesky"][k]
        assert np.abs(x - z["x"][k]).max() <= 1e-8 * max(1.0, np.abs(z["x"][k]).max())
        assert flops > 0


def test_device_code_matches_oracle_on_fresh_seed(emu, oracle, oracle_qp):
    sc = S.make(160, mode_mix=(0.34, 0.33, 0.33), pushes=True, terrain=True, seed=1234)
    got = emu.cycle(sc)
    ref, _ = oracle.run_cycle_batch(sc, nthreads=8, solver=oracle_qp)
    util.check_cycle_parity(got, ref, what="seed 1234")


def test_qp_record_against_oracle_stages(emu, oracle):
    """The compact QP record (front kernel -> solver kernel) stage by stage against the oracle's update()."""
    sc = S.make(8, mode_mix=(0.34, 0.33, 0.33), pushes=True, seed=77)
    rec = emu.cycle(sc)["rec"]
    for i in range(8):
        d = oracle.update_only(sc, i)
        Mcom = np.array(d.Mcom).reshape(18, 18)
        assert np.abs(rec[i, 0:36].reshape(6, 6) - Mcom[:6, :6]).max() < 1e-12
        assert np.abs(rec[i, 54:198].reshape(12, 12) - Mcom[6:, 6:]).max() < 1e-13
        assert np.abs(rec[i, 36:54] - np.array(d.hcom)).max() < 1e-11
        J = np.hstack([rec[i, 198:270].reshape(12, 6), rec[i, 270:414].reshape(12, 12)])
        assert np.abs(J - np.array(d.Jcom_lin).reshape(12, 18)).max() < 1e-13
        assert np.abs(rec[i, 414:426] - np.array(d.Jdqdcom_lin)).max() < 1e-12


def test_failure_is_reported_not_swallowed(emu):
    """Non-positive diagonal of Q -> ALGLIB throws (opt.cpp:48178-48181) and the reference swallows it
    (lopt.cpp:114-116); here it surfaces as a negative termination code."""
    z = np.load(util.GOLDEN + "/qp_stance.npz")
    Q = z["Q"][0].copy()
    Q[3, 3] = 0.0
    _, ist, _ = emu.qp_solve(Q, z["c"][0], z["L"][0], int(z["neq"]))
    assert ist[0] == -9


def test_multiplier_update_cache_is_exact(emu):
    """The reduced multiplier update reuses W, S = WW' and the factors while the active set is unchanged; a build that
    always recomputes (-DWBC_NO_REUSE) must give the same bits, and the cache must actually be hit."""
    import ctypes as C
    import os
    import subprocess
    so = os.path.join(util.EMU_DIR, "libwbc_emu_noreuse.so")
    src = os.path.join(util.EMU_DIR, "wbc_emu.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-DWBC_NO_REUSE", "-o", so, src])
    plain = util.Emu()
    plain.lib = C.CDLL(so)
    sc = S.make(300, mode_mix=(0.34, 0.33, 0.33), pushes=True, terrain=True, seed=4321)
    a, b = emu.cycle(sc), plain.cycle(sc)
    for k in ("tau", "w", "x", "qp_obj", "status"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["qp_info"][0], b["qp_info"][0])
    assert np.mean((a["qp_info"][5] & 64) != 0) > 0.9 and not ((b["qp_info"][5] & 64) != 0).any()


def test_staged_solver_reproduces_the_monolithic_one(emu, monkeypatch):
    """solve_stage_setup / _qloop / _update (the stages the solver kernel hands from warp to warp, state through the solve's
    global block) against solve_denseaul on the same instances: every output bit for bit, same counters."""
    sc = S.make(300, mode_mix=(0.34, 0.33, 0.33), pushes=True, terrain=True, seed=2468)
    a = emu.cycle(sc)
    monkeypatch.setenv("WBC_EMU_STAGED", "1")
    b = emu.cycle(sc)
    for k in ("tau", "w", "x", "qp_obj", "status"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["qp_info"], b["qp_info"])
