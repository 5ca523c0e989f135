"""Small mixed batch (stance + both swing modes, terrain, pushes) + trajectory sampling + the three plant steps + the observer forms and
the foot-wrench map, for compute-sanitizer.  WBC_SOLVER=mono|staged and WBC_FRONT=leg|thread select the kernels."""
import sys, numpy as np
sys.path.insert(0, ".")
from wbc_quadruped_dob_b200 import api, scenarios as S
n = int(sys.argv[1]) if len(sys.argv) > 1 else 96
sc = S.make(n, mode_mix=(0.3, 0.35, 0.35), pushes=True, terrain=True, seed=77)
p = api.default_params()
p.obs_order, p.obs_gain2 = 2, 4.0
b = api.WbcBatch(max_batch=n, device=0, params=p)
b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
for it in range(2):
    out = b.cycle(sc, want=("x", "qp_obj", "status", "qp_info", "qp_flops", "w3"))
tr = S.make_trajectory(sc, nseg=3, seed=3)
b.set_trajectory(tr)
b.sample_trajectory(n, t=tr["t"])
out2 = b.cycle({k: v for k, v in sc.items() if k not in api.TRAJ_FIELDS}, sampled_traj=True)
# forward-dynamics plant on host arrays (advanced in place), then the momentum plant
st = {k: np.array(sc[k], dtype=np.float64, order="C") for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
st["foot_force"] = np.zeros((12, n)); st["mode"] = np.ascontiguousarray(sc["mode"], dtype=np.int32)
b.plant_dynamics_step(st, out2["tau"], np.zeros((6, n)), substeps=3, gamma=100.0, diag=np.zeros((2, n)))
# contact plant on the same states, ground planes 1 mm below the feet
_, feet = S.forward_kinematics(st["base_pos"], st["base_rot"], st["q"])
cst = np.zeros(n, np.int32)
b.plant_contact_step(st, out2["tau"], np.zeros((6, n)), ground_z=feet[:, :, 2].T - 1e-3, substeps=3, contact=np.zeros((4, n), np.int32),
                     diag=np.zeros((4, n)), status=cst)
print("status ok:", bool((out["status"] == 0).all()), "flags", np.unique(out["qp_info"][5]), "finite",
      bool(np.isfinite(out2["tau"]).all() and np.isfinite(out["w3"]).all() and np.isfinite(st["q"]).all()), "contact plant ok:", bool((cst == 0).all()))
b.close()
