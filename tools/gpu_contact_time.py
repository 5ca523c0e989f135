"""Time per control period of the contact plant (wbc_plant_contact_step, five substeps), of its terrain form
(wbc_plant_contact_step_terrain) and of the bilateral forward-dynamics plant (wbc_plant_dynamics_step) on the same states, device
pointers, CUDA events around 20 calls of each after 3 warm-up calls, the three plants called in turn.  The states are a stance /
swing mix whose feet stand on, above and up to 3 mm below per-foot ground planes, under random torques and pushes (the mixed states
of tests/test_contact_plant.py), so that every kind of contact solve occurs; the terrain form gets the same gaps, measured along
per-foot normals up to 15 deg from vertical, and each foot's mu the instance's.  Each timed call starts from the same state.
Prints the GPU's name and power limit with the numbers."""
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from wbc_quadruped_dob_b200 import api, scenarios as S  # noqa: E402

STATE = ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
dev = torch.device("cuda", 0)
for n in (4096, 65536):
    rng = np.random.default_rng(5)
    sc = S.make(n, mode_mix=(0.4, 0.3, 0.3), pushes=False, seed=5)
    _, feet = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
    gap = rng.choice([-0.003, 0.0, 0.001, 0.004], size=(4, n)) * rng.uniform(0.0, 1.0, (4, n))
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    init = {k: T(sc[k]) for k in STATE}
    init["foot_force"] = torch.zeros(12, n, dtype=torch.float64, device=dev)
    init["mode"] = T(sc["mode"].astype(np.int32))
    din = {k: v.clone() for k, v in init.items()}
    tau, push = T(rng.normal(0.0, 4.0, (12, n))), T(rng.normal(0.0, 15.0, (6, n)))
    mu_h = rng.uniform(0.05, 1.0, n)
    gz, mu = T(feet[:, :, 2].T - gap), T(mu_h)
    ct = rng.uniform(np.cos(np.deg2rad(15.0)), 1.0, (4, n))
    ph = rng.uniform(0.0, 2 * np.pi, (4, n))
    tr_h, d_h = S.terrain_frames(np.stack([np.sqrt(1 - ct * ct) * np.cos(ph), np.sqrt(1 - ct * ct) * np.sin(ph), ct], axis=1), mu_h, feet)
    tr, pd = T(tr_h), T(d_h - gap)
    diag = torch.zeros(4, n, dtype=torch.float64, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    b = api.WbcBatch(max_batch=n)
    ts = torch.cuda.Stream()                            # the copies, the events and the plant on one (non-default) stream
    s = ts.cuda_stream
    plants = {
        "contact": lambda: b.plant_contact_step(din, tau, push, ground_z=gz, mu=mu, n=n, ld=n, substeps=5, diag=diag, status=status, stream=s, sync=False),
        "terrain": lambda: b.plant_contact_step(din, tau, push, terrain=tr, plane_d=pd, n=n, ld=n, substeps=5, diag=diag, status=status, stream=s,
                                                sync=False),
        "bilateral": lambda: b.plant_dynamics_step(din, tau, push, n=n, ld=n, substeps=5, gamma=100.0, stream=s, sync=False),
    }
    torch.cuda.synchronize()
    ms, wall, extra = {k: [] for k in plants}, {k: [] for k in plants}, {}
    for it in range(23):
        for name, call in plants.items():
            with torch.cuda.stream(ts):
                for k in init:
                    din[k].copy_(init[k])
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ts.synchronize()
                t0 = time.perf_counter()
                e0.record(ts); call(); e1.record(ts)
            torch.cuda.synchronize()
            if it >= 3:
                ms[name].append(e0.elapsed_time(e1))
                wall[name].append(1e3 * (time.perf_counter() - t0))
            if name != "bilateral" and it == 22:
                dg, st = diag.cpu().numpy(), status.cpu().numpy()
                extra[name] = ", failed %d, dual steps per robot-period %.2f (max %d), max KKT residual %.1e" % (
                    int((st != 0).sum()), dg[3].mean(), int(dg[3].max()), dg[2].max())
    for name in plants:
        print("n %6d %-9s plant, 5 substeps: median %.3f ms per control period (min %.3f, max %.3f; host clock to the synchronise %.3f ms)%s"
              % (n, name, np.median(ms[name]), min(ms[name]), max(ms[name]), np.median(wall[name]), extra.get(name, "")))
    print("n %6d terrain / flat contact plant: %.3f (median of the per-call ratios)" % (n, np.median(np.array(ms["terrain"]) / np.array(ms["contact"]))))
    b.close()
