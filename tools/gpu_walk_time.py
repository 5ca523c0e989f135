"""Time per control period of the walking loop at 4096 and 65 536 robots: the device loop wbc_gait_step -> wbc_cycle ->
wbc_plant_contact_step (five substeps), all enqueued on one stream without a host round trip, walking to commands on the test grid
(vx, vy, omega) and then trotting in place (cmd = None); the gait kernel alone; the controller and the plant alone (the device work
either loop does); and the host-driven trot-in-place loop of tests/test_contact_plant.py on the same states (contact flags copied to
the host every cycle, the base pose and joints copied to the host and forward kinematics run there at every phase start, the swing
targets built in numpy and copied back).  Device timings: CUDA events around each of 30 consecutive periods after a warm-up (60
periods walking, 120 in place so that the robots stop), median.  Host loop: wall clock around each of 92 periods (two phases), each
ending in a synchronisation, median and mean (the mean carries the phase starts' kinematics).  Flat ground, controller as in
tests/test_gait.py.  Prints the GPU's name and power limit with the numbers."""
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from tests.test_fdyn_plant import trot_in_place_targets  # noqa: E402
from tests.test_gait import _standing, api_params  # noqa: E402
from wbc_quadruped_dob_b200 import api, scenarios as S  # noqa: E402

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
dev = torch.device("cuda", 0)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
for n in (4096, 65536):
    sc, feet = _standing(n, 91)
    sc["base_pos"] = sc["base_pos"] - np.array([[0.0], [0.0], [1.0]]) * feet[:, :, 2].min(axis=1)[None]
    g = np.arange(n)
    cmd = T(np.vstack([np.linspace(-0.1, 0.1, 16)[g % 16], np.linspace(-0.05, 0.05, 16)[(g // 16) % 16], np.linspace(-0.2, 0.2, 16)[(g // 256) % 16]]))
    din = {k: T(v) for k, v in sc.items() if isinstance(v, np.ndarray)}
    din["mode"] = torch.zeros(n, dtype=torch.int32, device=dev)
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    zero = torch.zeros(6, n, dtype=torch.float64, device=dev)
    contact = torch.zeros(4, n, dtype=torch.int32, device=dev)
    b = api.WbcBatch(max_batch=n, params=api_params())
    b.set_observer_state(np.zeros((6, n)), np.zeros((6, n)))
    gs = b.gait_state(n, device=dev)
    ts = torch.cuda.Stream()
    ts.wait_stream(torch.cuda.current_stream())               # the tensors above were filled on the default stream
    s = ts.cuda_stream
    b.gait_init(din, gs, T(np.random.default_rng(1).integers(0, 184, n).astype(np.int32)))
    gait = lambda: b.gait_step(din, gs, cmd, contact, out=din, stream=s, sync=False)
    trot = lambda: b.gait_step(din, gs, None, contact, out=din, stream=s, sync=False)
    rest = [lambda: b.cycle_device(din, dout, n, n, stream=s, sync=False),
            lambda: b.plant_contact_step(din, dout["tau"], zero, n=n, ld=n, substeps=5, contact=contact, stream=s, sync=False)]
    torch.cuda.synchronize()

    def events(calls, periods):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(periods + 1)]
        with torch.cuda.stream(ts):
            ev[0].record(ts)
            for k in range(periods):
                for f in calls:
                    f()
                ev[k + 1].record(ts)
        ts.synchronize()
        return np.array([ev[k].elapsed_time(ev[k + 1]) for k in range(periods)])
    events([gait] + rest, 60)
    loop = events([gait] + rest, 30)
    alone = events([gait], 30)
    # the same loop trotting in place (cmd = None), the host loop's kind of work; after a warm-up in which the robots stop
    events([trot] + rest, 120)
    inplace = events([trot] + rest, 30)
    work = events(rest, 30)                           # controller + plant alone on those states: the device work of either loop
    # host-driven loop (tests/test_contact_plant.py): schedule and touchdown on the host, targets built there
    P, sched = 46, [S.MODE_STANCE, S.MODE_SWING_BR_FL, S.MODE_STANCE, S.MODE_SWING_BL_FR]
    wall, anchor, landed = [], None, None
    torch.cuda.synchronize()
    with torch.cuda.stream(ts):
        for c in range(2 * P + 1):
            t0 = time.perf_counter()
            mode, sph = sched[(c // P) % 4], (c % P) / P
            first, second = (1, 3) if mode == S.MODE_SWING_BL_FR else (0, 2)
            if c % P == 0:
                host = {k: din[k].cpu().numpy() for k in ("base_pos", "base_rot", "q")}
                _, anchor = S.forward_kinematics(host["base_pos"], host["base_rot"], host["q"])
                landed = np.zeros(n, bool)
            if mode != S.MODE_STANCE:
                cf = contact.cpu().numpy()
                landed |= (sph > 0.5) & (cf[first] > 0) & (cf[second] > 0)
                m = np.where(landed, S.MODE_STANCE, mode).astype(np.int32)
            else:
                m = np.full(n, mode, np.int32)
            din["mode"].copy_(torch.from_numpy(m))
            sp, sv, sa = trot_in_place_targets(anchor, mode, sph, P * 0.0025, 0.03)
            din["sw_des_pos"].copy_(torch.from_numpy(sp)); din["sw_des_vel"].copy_(torch.from_numpy(sv)); din["sw_des_acc"].copy_(torch.from_numpy(sa))
            for f in rest:
                f()
            ts.synchronize()
            if c > 0:
                wall.append(1e3 * (time.perf_counter() - t0))
    wall = np.array(wall)
    print("n=%d: device loop walking (gait + cycle + contact plant, 5 substeps) %.3f ms/period (median of 30; min %.3f, max %.3f); gait kernel "
          "alone %.4f ms; device loop trotting in place %.3f ms/period (min %.3f); cycle + contact plant alone %.3f ms; host-driven trot in "
          "place %.3f ms/period median, %.3f mean (92 periods)"
          % (n, np.median(loop), loop.min(), loop.max(), np.median(alone), np.median(inplace), inplace.min(), np.median(work), np.median(wall),
             wall.mean()))
    b.close()
