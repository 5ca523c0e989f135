"""Parity of the CUDA path (through the C ABI) with the CPU oracle.  Everything here needs a real B200."""
import numpy as np
import pytest

from tests import util
from wbc_quadruped_dob_b200 import api
from wbc_quadruped_dob_b200 import scenarios as S

pytestmark = pytest.mark.gpu


def _run(batch, sc):
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    return batch.cycle(sc)


@pytest.mark.parametrize("name", ["cycle_standing", "cycle_trot_pushes", "cycle_mixed_terrain"])
def test_cycle_matches_golden(gpu_batch, name):
    sc, gold = util.load_golden(name)
    n = sc["mode"].shape[0]
    got = _run(gpu_batch, sc)
    util.check_cycle_parity(got, gold, what=name)
    yd, yw = gpu_batch.get_observer_state(n)
    assert np.abs(yd.T - gold["yd"]).max() <= util.TOL_OBS
    assert np.abs(yw.T - gold["yw"]).max() <= util.TOL_OBS
    assert np.abs(got["x"].T - gold["x"]).max() <= 1e-7 * max(1.0, np.abs(gold["x"]).max())
    assert np.mean(got["qp_info"][0] == gold["ncholesky"]) >= 0.97
    assert gpu_batch.last_launches() == 2


def test_trot_replay_single_robot_chained_observer(gpu_batch):
    """BASELINE config 1: ONE DogBot, cycle after cycle, observer state carried inside the ctx."""
    sc, gold = util.load_golden("cycle_trot_replay")
    n = sc["mode"].shape[0]
    gpu_batch.set_observer_state(np.zeros((6, 1)), np.zeros((6, 1)))
    for i in range(n):
        one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
        got = gpu_batch.cycle(one)
        assert np.abs(got["w"][:, 0] - gold["w"][i]).max() <= util.TOL_OBS * max(1.0, np.abs(gold["w"][i]).max())
        assert util.rel_rows(got["tau"].T, gold["tau"][i:i + 1]).max() <= util.TOL_TAU


@pytest.mark.parametrize("cfg,n", [("standing_4096", 4096), ("trot_65536", 3000), ("mixed_terrain_1m", 3000)])
def test_cycle_matches_oracle_on_baseline_configs(gpu_batch, oracle, oracle_qp, cfg, n):
    sc = S.make_config(cfg, n=n)
    got = _run(gpu_batch, sc)
    ref, _ = oracle.run_cycle_batch(sc, nthreads=16, solver=oracle_qp)
    worst = util.check_cycle_parity(got, ref, what=cfg)
    print(cfg, "worst torque rel err", worst)


def test_dispatch_order_never_changes_a_result(gpu_batch):
    """The work queue hands out instances longest-first from the second cycle on (WBC_FIFO_DISPATCH turns that off):
    every output must be bit-identical whichever order the warps took the instances in, and the order the front kernel
    builds must be a permutation (a lost or duplicated ticket would leave a stale or doubly written torque)."""
    sc = S.make(3000, mode_mix=(0.4, 0.3, 0.3), pushes=True, seed=91)
    want = ("x", "qp_obj", "status", "qp_info")
    gpu_batch.fifo_dispatch = True
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    first = gpu_batch.cycle(sc, want=want)
    gpu_batch.fifo_dispatch = False
    for _ in range(3):      # cycles 2.. use the durations recorded by the cycle before
        gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        again = gpu_batch.cycle(sc, want=want)
        for k in ("tau", "w", "x", "qp_obj", "status", "qp_info"):
            assert np.array_equal(first[k], again[k]), k
    # a different batch size right after: the stale order is not used
    sub = {k: (np.ascontiguousarray(v[..., :1000]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    gpu_batch.set_observer_state(sub["obs_yd"], sub["obs_yw"])
    part = gpu_batch.cycle(sub, want=want)
    assert np.array_equal(part["tau"], first["tau"][:, :1000])


def test_update_stages_match_oracle(gpu_batch, oracle):
    sc = S.make(64, mode_mix=(0.34, 0.33, 0.33), pushes=True, seed=77)
    dbg = gpu_batch.debug_update(sc)
    for i in range(0, 64, 7):
        d = oracle.update_only(sc, i)
        assert np.abs(dbg["M"][:, i] - np.array(d.M)).max() < 1e-12
        assert np.abs(dbg["h"][:, i] - np.array(d.h)).max() < 1e-11
        assert np.abs(dbg["g"][:, i] - np.array(d.g)).max() < 1e-11
        assert np.abs(dbg["Jac_lin"][:, i] - np.array(d.Jac_lin)).max() < 1e-13
        assert np.abs(dbg["Jdqd_lin"][:, i] - np.array(d.Jdqd_lin)).max() < 1e-12
        assert np.abs(dbg["com"][:, i] - np.array(d.com)).max() < 1e-13
        assert np.abs(dbg["com_vel"][:, i] - np.array(d.com_vel)).max() < 1e-13
        Mcom = np.array(d.Mcom).reshape(18, 18)
        assert np.abs(dbg["Mcom_b"][:, i].reshape(6, 6) - Mcom[:6, :6]).max() < 1e-12
        assert np.abs(dbg["Mcom_j"][:, i].reshape(12, 12) - Mcom[6:, 6:]).max() < 1e-13
        assert np.abs(dbg["hcom"][:, i] - np.array(d.hcom)).max() < 1e-11
        assert np.abs(dbg["gcom"][:, i] - np.array(d.gcom)).max() < 1e-11
        assert np.abs(dbg["Jcom_lin"][:, i] - np.array(d.Jcom_lin)).max() < 1e-13
        assert np.abs(dbg["Jdqdcom_lin"][:, i] - np.array(d.Jdqdcom_lin)).max() < 1e-12
        assert np.abs(dbg["foot_pos"][:, i] - np.array(d.foot_pos)).max() < 1e-13
        assert np.abs(dbg["foot_vel"][:, i] - np.array(d.foot_vel)).max() < 1e-13


@pytest.mark.parametrize("name", ["qp_stance", "qp_swing"])
def test_opt_operator_matches_reference_alglib_golden(gpu_batch, name):
    """OPT::opt_stance / opt_swing (lopt.cpp:84-154): dense (Q, c, L) in, x out, against the reference's own outputs."""
    z = np.load(util.GOLDEN + "/" + name + ".npz")
    x, status, info, flops = gpu_batch.qp_solve(z["Q"], z["c"], z["L"], int(z["neq"]))
    assert (status == 0).all()
    assert np.array_equal(info[:, 0], z["ncholesky"])
    assert np.abs(x - z["x"]).max() <= 1e-8 * max(1.0, np.abs(z["x"]).max())
    assert (flops > 0).all()


def test_opt_class_mirror(gpu_batch):
    z = np.load(util.GOLDEN + "/qp_stance.npz")
    opt = api.OPT(30, 86, 82, batch=gpu_batch)
    opt.setQ(z["Q"][0]); opt.setc(z["c"][0]); opt.setL_stance(z["L"][0])
    x = opt.opt_stance()
    assert np.abs(x - z["x"][0]).max() <= 1e-8 * max(1.0, np.abs(z["x"][0]).max())
    zs = np.load(util.GOLDEN + "/qp_swing.npz")
    opt.setQ(zs["Q"][1]); opt.setc(zs["c"][1]); opt.setL_swing(zs["L"][1])
    x = opt.opt_swing()
    assert np.abs(x - zs["x"][1]).max() <= 1e-8 * max(1.0, np.abs(zs["x"][1]).max())


def test_solver_failure_is_reported(gpu_batch):
    z = np.load(util.GOLDEN + "/qp_stance.npz")
    Q = z["Q"][:2].copy()
    Q[1, 3, 3] = 0.0          # ALGLIB throws on a non-positive diagonal with autodiag scaling (opt.cpp:48178-48181)
    x, status, _, _ = gpu_batch.qp_solve(Q, z["c"][:2], z["L"][:2], int(z["neq"]))
    assert status[0] == 0 and status[1] == -9


def test_edge_cases_empty_single_and_ragged(gpu_batch, oracle, oracle_qp):
    sc = S.make(0)
    out = gpu_batch.cycle(sc, n=0)
    assert out["tau"].shape == (12, 0)
    sc = S.make(37, mode_mix=(0.3, 0.3, 0.4), pushes=True, seed=5)
    ref, _ = oracle.run_cycle_batch(sc, nthreads=4, solver=oracle_qp)
    # ragged: n smaller than the arrays' leading dimension
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    got = gpu_batch.cycle(sc, n=21)
    util.check_cycle_parity(got, {k: v[:21] for k, v in ref.items()}, what="ragged")
    one = {k: (v[..., 36:37] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    gpu_batch.set_observer_state(one["obs_yd"], one["obs_yw"])
    got = gpu_batch.cycle(one)
    util.check_cycle_parity(got, {k: v[36:37] for k, v in ref.items()}, what="single")
    with pytest.raises(api.WbcError):
        gpu_batch.cycle(S.make(8), n=gpu_batch.max_batch + 1)


def test_observer_disabled_reproduces_shipped_reference(gpu_batch, oracle, oracle_qp):
    """The shipped binary never calls estimate() (main.cpp:1029): w = 0 and the state does not move."""
    sc = S.make(64, mode_mix=(0.5, 0.25, 0.25), seed=8)
    p = api.default_params()
    p.observer_enabled = 0
    gpu_batch.set_params(p)
    try:
        got = _run(gpu_batch, sc)
        yd, yw = gpu_batch.get_observer_state(64)
    finally:
        gpu_batch.set_params(api.default_params())
    ref, _ = oracle.run_cycle_batch(sc, params=oracle.default_params(observer_enabled=0), nthreads=4, solver=oracle_qp)
    util.check_cycle_parity(got, ref, what="observer off")
    assert np.all(got["w"] == 0.0) and np.array_equal(yd, sc["obs_yd"]) and np.array_equal(yw, sc["obs_yw"])


def test_full_size_properties_65536(gpu_batch):
    """BASELINE config 3 at full size: size-independent properties instead of the (slow) oracle."""
    n = 65536
    sc = S.make_config("trot_65536", n=n)
    got = _run(gpu_batch, sc)
    assert (got["status"] == 0).all()
    assert np.isfinite(got["tau"]).all() and np.isfinite(got["w"]).all()
    # determinism: same inputs, same bits
    again = _run(gpu_batch, sc)
    assert np.array_equal(got["tau"], again["tau"]) and np.array_equal(got["x"], again["x"])
    # shard invariance: instances are independent, so solving a slice alone gives the same bits
    lo, hi = 30000, 34096
    part = {k: (np.ascontiguousarray(v[..., lo:hi]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    sub = _run(gpu_batch, part)
    assert np.array_equal(sub["tau"], got["tau"][:, lo:hi])
    # stance QPs converge (SURVEY App. F): equality rows hold, friction cones and torque limits respected
    st = sc["mode"] == 0
    x = got["x"][:, st]
    fz = x[[20, 23, 26, 29]]
    assert fz.min() > -1e-3
    assert np.abs(got["tau"][:, st]).max() <= 60.0 * (1 + 1e-3)
    mu = 0.6
    for f in range(4):
        assert (np.abs(x[18 + 3 * f]) <= mu * x[20 + 3 * f] + 1e-2).all()
        assert (np.abs(x[19 + 3 * f]) <= mu * x[20 + 3 * f] + 1e-2).all()


def test_device_pointer_path_with_torch(gpu_batch):
    torch = pytest.importorskip("torch")
    n = 512
    sc = S.make(n, mode_mix=(0.3, 0.35, 0.35), pushes=True, seed=31)
    host = _run(gpu_batch, sc)
    dev_in = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in sc.items() if isinstance(v, np.ndarray)}
    dev_out = {"tau": torch.zeros(12, n, dtype=torch.float64, device="cuda"), "w": torch.zeros(6, n, dtype=torch.float64, device="cuda"),
               "x": torch.zeros(30, n, dtype=torch.float64, device="cuda")}
    torch.cuda.synchronize()
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    gpu_batch.cycle_device(dev_in, dev_out, n, n, stream=torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(dev_out["tau"].cpu().numpy(), host["tau"])
    assert np.array_equal(dev_out["w"].cpu().numpy(), host["w"])


def test_page_locked_arrays_take_the_direct_copy_path_with_identical_results(gpu_batch):
    """wbc_host_alloc'ed SoA arrays are DMA'd directly (no bounce buffer); results are bit-identical to the pageable
    path, with a padded leading dimension (ld > n) and preallocated page-locked outputs."""
    sc, gold = util.load_golden("cycle_trot_pushes")
    n = sc["mode"].shape[0]
    ref = _run(gpu_batch, sc)
    ld = n + 7
    pin = {}
    for k, v in sc.items():
        if not isinstance(v, np.ndarray) or k in ("obs_yd", "obs_yw"):
            pin[k] = v
            continue
        shape = (v.shape[0], ld) if v.ndim == 2 else (ld,)
        a = gpu_batch.pinned(shape, v.dtype)
        a[...] = 0
        a[..., :n] = v
        pin[k] = a
    out = {"tau": gpu_batch.pinned((12, n)), "w": gpu_batch.pinned((6, n)), "x": gpu_batch.pinned((30, n)), "qp_obj": gpu_batch.pinned((n,))}
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    got = gpu_batch.cycle(pin, n=n, out=out)
    for k in ("tau", "w", "x", "qp_obj"):
        assert np.array_equal(got[k], ref[k]), k
    util.check_cycle_parity({**got, "status": ref["status"]}, gold, what="pinned")


def test_last_solve_cycles_reports_every_instance(gpu_batch):
    sc, _ = util.load_golden("cycle_standing")
    n = sc["mode"].shape[0]
    _run(gpu_batch, sc)
    cyc = gpu_batch.last_solve_cycles(n)
    assert cyc.shape == (n,) and (cyc > 0).all() and (cyc < 2e9).all()


def test_full_size_properties_config4_shard_131072():
    """BASELINE config 4's per-GPU shard (1 M instances over 8 GPUs = 131 072 each, mixed gaits, rough terrain) through
    size-independent properties: permutation equivariance (reversing the instance order reverses the outputs bit for
    bit although the work queue, the longest-first order and the warp that solves each instance all change), and the
    friction pyramids of the stance instances in their own per-foot terrain frames."""
    n = 131072
    sc = S.make_config("mixed_terrain_1m", n=n)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        got = _run(b, sc)
        assert (got["status"] == 0).all()
        assert np.isfinite(got["tau"]).all() and np.isfinite(got["w"]).all()
        rev = {k: (np.ascontiguousarray(v[..., ::-1]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
        got_r = _run(b, rev)
        for k in ("tau", "w", "x"):
            assert np.array_equal(got_r[k][:, ::-1], got[k]), k
        st = sc["mode"] == 0
        x, T = got["x"][:, st], sc["terrain"][:, st]
        assert np.abs(got["tau"][:, st]).max() <= 60.0 * (1 + 1e-3)
        for f in range(4):
            fv = x[18 + 3 * f:21 + 3 * f]
            nn, t1, t2, mu = T[10 * f:10 * f + 3], T[10 * f + 3:10 * f + 6], T[10 * f + 6:10 * f + 9], T[10 * f + 9]
            fn = (nn * fv).sum(axis=0)
            assert fn.min() > -1e-3
            assert (np.abs((t1 * fv).sum(axis=0)) <= mu * fn + 1e-2).all()
            assert (np.abs((t2 * fv).sum(axis=0)) <= mu * fn + 1e-2).all()
    finally:
        b.close()


def test_config4_whole_on_one_gpu_equals_its_shards():
    """Maximum size: ALL 1 048 576 instances of BASELINE config 4 in one batch on one GPU (the configuration names 8 GPUs; one has the
    memory for it).  Every instance is solved, and what a rank of the 8-GPU run computes for its shard -- the same instances
    generated from their offset, solved in a batch of 131 072 -- is bit for bit what the whole batch gives at those indices:
    sharding changes who computes an instance and with which neighbours, nothing else."""
    n = 1 << 20
    sc = S.make_config("mixed_terrain_1m", n=n)
    b = api.WbcBatch(max_batch=n, device=0)
    try:
        got = _run(b, sc)
        assert (got["status"] == 0).all()
        assert np.isfinite(got["tau"]).all() and np.isfinite(got["w"]).all()
        assert np.abs(got["tau"][:, sc["mode"] == 0]).max() <= 60.0 * (1 + 1e-3)
    finally:
        b.close()
    for rank in (0, 5):
        lo = rank * 131072
        part = S.make_config("mixed_terrain_1m", n=131072, start=lo)
        for k in ("q", "base_vel", "terrain", "mode"):
            assert np.array_equal(part[k], sc[k][..., lo:lo + 131072]), k          # the generator is offset-addressable
        bs = api.WbcBatch(max_batch=131072, device=0)
        try:
            sub = _run(bs, part)
        finally:
            bs.close()
        for k in ("tau", "w", "x"):
            assert np.array_equal(sub[k], got[k][:, lo:lo + 131072]), (rank, k)
