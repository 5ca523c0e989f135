"""BASELINE config 5: disturbance-rejection sweep (push direction x magnitude x observer gain x state), closed through the
synthetic CoM-momentum plant (wbc_plant_step; stands in for Gazebo + force_plugin's ModelPush, fp.cpp:124-491)."""
import numpy as np
import pytest

from tests import util
from wbc_quadruped_dob_b200 import scenarios as S

SMALL = dict(directions=2, magnitudes=(20.0, 80.0), gains=(10.0, 50.0, 200.0), states=2)


def _copy(sc):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sc.items()}


def test_sweep_grid_layout():
    sc = S.push_sweep(n=None, **SMALL)
    n = sc["mode"].shape[0]
    assert n == 2 * 2 * 3 * 2
    d, m, g, s = sc["grid"]
    assert (np.arange(n) == ((d * 2 + m) * 3 + g) * 2 + s).all()
    assert (sc["mode"] == S.MODE_STANCE).all() and not sc["dq"].any() and not sc["base_vel"].any()
    assert np.allclose(np.linalg.norm(sc["push"][:3], axis=0), np.array([20.0, 80.0])[m])
    assert set(np.unique(sc["obs_gain"])) == {10.0, 50.0, 200.0}
    # a slice of the grid equals the same rows of the full grid (rank sharding)
    part = S.push_sweep(n=7, start=5, **SMALL)
    for k in ("q", "push", "base_pos", "foot_force"):
        assert np.array_equal(part[k], sc[k][..., 5:12])
    assert np.array_equal(part["obs_gain"], sc["obs_gain"][5:12])
    full = S.push_sweep(n=4, start=262140)
    assert full["mode"].shape[0] == 4 and full["grid"][:, -1].tolist() == [15, 7, 7, 255]


def test_oracle_closed_loop_rejects_the_push(oracle, oracle_qp):
    """Observer estimate converges to the injected wrench like exp(-k t) (main.cpp:707-719 is a first-order filter with
    gain k), faster for larger k, and the closed loop stays bounded."""
    sc = S.push_sweep(n=None, **SMALL)
    cur = _copy(sc)
    P = oracle.default_params()
    push = sc["push"].T
    scale = np.abs(push).max(axis=1)
    err = []
    for it in range(120):
        res, _ = oracle.run_cycle_batch_gains(cur, P, nthreads=8, solver=oracle_qp)
        assert (res["status"] == 0).all()
        err.append(np.abs(res["w"] - push).max(axis=1) / scale)
        pos, vel, ff = oracle.plant_step(cur, cur["push"], x=res["x"], params=P)
        cur["base_pos"], cur["base_vel"], cur["foot_force"] = pos, vel, ff
        cur["obs_yd"], cur["obs_yw"] = np.ascontiguousarray(res["yd"].T), np.ascontiguousarray(res["yw"].T)
        assert np.abs(vel[:3]).max() < 1.0 and np.abs(vel[3:]).max() < 6.0   # orientation is frozen: only damping acts on omega
    err = np.array(err)                       # [cycle, instance]
    g = sc["obs_gain"]
    t = 0.0025 * 119
    for k in (10.0, 50.0, 200.0):
        e = err[-1, g == k]
        assert (e < 3.0 * np.exp(-k * t / (1 + k * 0.0025)) + 1e-9).all(), (k, e.max())
    # rise time (first cycle with error below 1/e) shrinks with the gain
    rise = np.array([np.argmax(err[:, i] < np.exp(-1.0)) for i in range(err.shape[1])])
    assert rise[g == 10.0].min() > rise[g == 50.0].max() > rise[g == 200.0].max() >= 1


@pytest.mark.gpu
def test_sweep_rollout_matches_oracle_every_cycle(gpu_batch, oracle, oracle_qp):
    """GPU closed loop (wbc_cycle + wbc_plant_step, per-instance observer gains, observer state kept in the ctx); the
    oracle is teacher-forced with the GPU's inputs each cycle.  w within 1e-9, torques 1e-6, plant state 1e-10."""
    sc = S.push_sweep(n=None, **SMALL)
    n = sc["mode"].shape[0]
    cur = _copy(sc)
    P = oracle.default_params()
    gpu_batch.set_observer_state(cur["obs_yd"], cur["obs_yw"])
    for it in range(40):
        got = gpu_batch.cycle(cur)
        ref, _ = oracle.run_cycle_batch_gains(cur, P, nthreads=8, solver=oracle_qp)
        util.check_cycle_parity(got, ref, what="sweep cycle %d" % it)
        yd, yw = gpu_batch.get_observer_state(n)
        assert np.abs(yd.T - ref["yd"]).max() <= util.TOL_OBS * max(1.0, np.abs(ref["yd"]).max())
        rpos, rvel, rff = oracle.plant_step(cur, cur["push"], x=got["x"].T, params=P)
        pos, vel, ff = cur["base_pos"].copy(), cur["base_vel"].copy(), cur["foot_force"].copy()
        gpu_batch.plant_step(pos, vel, cur["push"], foot_force=ff, x=got["x"])
        assert gpu_batch.last_launches() == 1
        assert np.abs(vel - rvel).max() <= 1e-10 and np.abs(pos - rpos).max() <= 1e-12
        assert np.abs(ff - rff).max() <= 1e-10 * max(1.0, np.abs(rff).max())
        cur["base_pos"], cur["base_vel"], cur["foot_force"] = pos, vel, ff
        cur["obs_yd"], cur["obs_yw"] = yd, yw
    # open-loop plant (measured forces) as well
    rpos, rvel, _ = oracle.plant_step(cur, cur["push"], params=P)
    gpu_batch.cycle(cur)
    pos, vel = cur["base_pos"].copy(), cur["base_vel"].copy()
    gpu_batch.plant_step(pos, vel, cur["push"])
    assert np.abs(vel - rvel).max() <= 1e-10 and np.abs(pos - rpos).max() <= 1e-12


@pytest.mark.gpu
def test_sweep_device_resident_rollout(gpu_batch):
    """The rollout with every buffer resident on the GPU (the path bench.py --workload push_sweep times) equals the
    host-pointer rollout bit for bit, and the estimate converges."""
    import torch
    sc = S.push_sweep(n=None, **SMALL)
    n = sc["mode"].shape[0]
    dev = torch.device("cuda", 0)
    cur = _copy(sc)
    gpu_batch.set_observer_state(cur["obs_yd"], cur["obs_yw"])
    host_w = []
    for it in range(30):
        got = gpu_batch.cycle(cur)
        gpu_batch.plant_step(cur["base_pos"], cur["base_vel"], cur["push"], foot_force=cur["foot_force"], x=got["x"])
        host_w.append(got["w"].copy())
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray) and k != "grid"}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "x": torch.zeros(30, n, dtype=torch.float64, device=dev)}
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    for it in range(30):
        gpu_batch.cycle_device(din, dout, n, n)
        gpu_batch.plant_step(din["base_pos"], din["base_vel"], din["push"], foot_force=din["foot_force"], x=dout["x"], n=n, ld=n)
        assert np.array_equal(dout["w"].cpu().numpy(), host_w[it])
    assert np.array_equal(din["base_vel"].cpu().numpy(), cur["base_vel"])
    w = dout["w"].cpu().numpy()
    fast = sc["obs_gain"] == 200.0
    assert (np.abs(w - sc["push"])[:, fast].max(axis=0) < 1e-3 * np.abs(sc["push"][:, fast]).max(axis=0)).all()
