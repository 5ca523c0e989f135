"""On-device trajectory sampling (SURVEY.md 8f-1): the oracle's restatement of towr::Spline::GetPoint (spline.cc:48-93,
polynomial.cc:50-104) against the cubic-Hermite interpolation properties, the device code (host build) against the
oracle, and -- on the GPU -- the kernel and the WBC_SAMPLED_TRAJ cycle against both."""
import numpy as np
import pytest

from tests import util
from wbc_quadruped_dob_b200 import scenarios as S

TOL = 1e-12      # relative, on positions / velocities / accelerations (the device uses t*t*t where the reference calls pow)
NAMES = ["com_des_pos", "com_des_vel", "com_des_acc", "sw_des_pos", "sw_des_vel", "sw_des_acc"]


def _close(a, b):
    return np.abs(a - b).max() <= TOL * max(1.0, np.abs(b).max())


def test_oracle_spline_interpolates_its_nodes_and_keeps_the_previous_polynomial_at_junctions(oracle):
    rng = np.random.default_rng(3)
    for nseg in (1, 2, 5, 8):
        dur = rng.uniform(0.1, 0.6, nseg)
        nodes = rng.normal(0, 1, (nseg + 1, 6))
        sid, p, v, a = oracle.spline_point(dur, nodes, 0.0)
        assert sid == 0 and np.array_equal(p, nodes[0, :3]) and np.array_equal(v, nodes[0, 3:])
        for j in range(nseg):
            tj = dur[:j + 1].sum()
            sid, p, v, _ = oracle.spline_point(dur, nodes, tj)
            assert sid == j                                   # "at junctions, returns previous spline" (spline.cc:59)
            assert np.abs(p - nodes[j + 1, :3]).max() < 1e-12 and np.abs(v - nodes[j + 1, 3:]).max() < 1e-11
            if j + 1 < nseg:
                sid2, p2, v2, _ = oracle.spline_point(dur, nodes, tj + 1e-6)
                assert sid2 == j + 1 and np.abs(p2 - p).max() < 1e-4
        # velocity is the derivative of position, acceleration of velocity (central differences inside a polynomial)
        t, h = 0.37 * dur[0], 1e-5
        _, pm, vm, _ = oracle.spline_point(dur, nodes, t - h)
        _, pp, vp, _ = oracle.spline_point(dur, nodes, t + h)
        _, _, v0, a0 = oracle.spline_point(dur, nodes, t)
        assert np.abs((pp - pm) / (2 * h) - v0).max() < 1e-6 and np.abs((vp - vm) / (2 * h) - a0).max() < 1e-5
        assert oracle.spline_point(dur, nodes, -1.0)[0] == -1 and oracle.spline_point(dur, nodes, dur.sum() + 1.0)[0] == -1


@pytest.mark.parametrize("nseg", [1, 3, 8])
def test_device_sampling_code_matches_oracle(emu, oracle, nseg):
    sc = S.make(64, mode_mix=(0.3, 0.35, 0.35), pushes=True, seed=21)
    tr = S.make_trajectory(sc, nseg=nseg, seed=5 + nseg)
    got = emu.sample_trajectory(tr, tr["t"])
    ref = oracle.sample_trajectory(tr, tr["t"])
    for k in NAMES:
        assert _close(got[k], ref[k]), k
    # t = 0 reproduces the plan's start = the scenario's own desired pose
    z = np.flatnonzero(tr["t"] == 0.0)
    assert len(z) and np.array_equal(got["com_des_pos"][:, z], sc["com_des_pos"][:, z])


@pytest.mark.gpu
def test_gpu_sampling_matches_oracle_and_feeds_the_cycle(gpu_batch, oracle, oracle_qp):
    n = 3000
    sc = S.make(n, mode_mix=(0.3, 0.35, 0.35), pushes=True, terrain=True, seed=33)
    tr = S.make_trajectory(sc, nseg=4, seed=9)
    gpu_batch.set_trajectory(tr)
    got = gpu_batch.sample_trajectory(n, t=tr["t"], fetch=True)
    ref = oracle.sample_trajectory(tr, tr["t"])
    for k in NAMES:
        assert _close(got[k], ref[k]), k
    assert gpu_batch.last_launches() == 1
    # the cycle fed from the device-resident samples == the cycle fed the same samples from the host, bit for bit
    sc_s = dict(sc)
    sc_s.update(got)
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    host = gpu_batch.cycle(sc_s)
    gpu_batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    gpu_batch.sample_trajectory(n, t=tr["t"])
    no_traj = {k: v for k, v in sc.items() if k not in NAMES}
    dev = gpu_batch.cycle(no_traj, sampled_traj=True)
    for k in ("tau", "w", "x"):
        assert np.array_equal(dev[k], host[k]), k
    # ... and agrees with the CPU controller run on the oracle's samples
    sc_o = dict(sc)
    sc_o.update(ref)
    want, _ = oracle.run_cycle_batch(sc_o, nthreads=8, solver=oracle_qp)
    util.check_cycle_parity(dev, want, what="sampled trajectory")


@pytest.mark.gpu
def test_gpu_sampling_uniform_time_and_errors(gpu_batch, oracle):
    from wbc_quadruped_dob_b200 import api
    sc = S.make(100, mode_mix=(1.0, 0.0, 0.0), seed=2)
    tr = S.make_trajectory(sc, nseg=2, seed=1)
    gpu_batch.set_trajectory(tr)
    got = gpu_batch.sample_trajectory(100, t_all=0.05, fetch=True)
    ref = oracle.sample_trajectory(tr, np.full(100, 0.05))
    for k in NAMES:
        assert _close(got[k], ref[k]), k
    with pytest.raises(api.WbcError):
        gpu_batch.sample_trajectory(101, t_all=0.0)          # more instances than the plan covers
    bad = dict(tr)
    bad["nseg"] = 9
    with pytest.raises(api.WbcError):
        gpu_batch.set_trajectory(bad)
