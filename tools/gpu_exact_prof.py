"""Per-phase profile of the exact-mode solver kernel (wbc_solve_exact_kernel<true>): SM cycles per phase of the Goldfarb-Idnani
solve, summed over every warp of one cycle, from clock64 counters (a ctx created with WBC_STAGE_PROF=1; the profiled kernel is a
separate instantiation, the shipped one carries no counters).  Workloads and inputs as bench.py.  Prints one JSON document.

    WBC_STAGE_PROF=1 python tools/gpu_exact_prof.py [--workloads standing_4096,trot_65536] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PHASES = ["assemble (record staging, validation, assembly)", "setup (scaling, Cholesky, J = L^-T, unconstrained minimiser)",
          "residual sweep over the inactive rows", "d = J'n (+ row load and value)", "z = J2 d2, r = R^-1 d1", "steps of y and u, t1",
          "add a row (Householder reflection on d and J, R column)", "drop a row (R column shift, Givens on R and J)", "torque map and outputs"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="standing_4096,trot_65536")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not os.environ.get("WBC_STAGE_PROF"):
        raise SystemExit("set WBC_STAGE_PROF=1: the counters are only kept by a ctx created with it")
    import torch
    from wbc_quadruped_dob_b200 import api
    from wbc_quadruped_dob_b200 import scenarios as S
    dev = torch.device("cuda", 0)
    clock_mhz = torch.cuda.get_device_properties(0).clock_rate / 1e3 if hasattr(torch.cuda.get_device_properties(0), "clock_rate") else None
    doc = {"gpu": torch.cuda.get_device_name(0), "kernel": "wbc_solve_exact_kernel<true> (clock64 counters per phase)", "workloads": []}
    for name in args.workloads.split(","):
        sc = S.make_config(name)
        n = int(sc["mode"].shape[0])
        b = api.WbcBatch(max_batch=n, device=0)
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
        dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
                "qp_info": torch.zeros(8, n, dtype=torch.int32, device=dev)}
        for _ in range(args.warmup + 1):
            b.cycle_device(din, dout, n, n, exact=True)
        torch.cuda.synchronize()
        front_ms, solve_ms = b.last_timing()
        rows = b.stage_profile().astype(np.float64)
        rows = rows[rows[:, 9] > 0]
        tot = rows[:, :9].sum(axis=0)
        solves, changes, kernel = rows[:, 9].sum(), rows[:, 10].sum(), rows[:, 11]
        busy = tot.sum()
        info = dout["qp_info"].cpu().numpy()
        doc["workloads"].append({
            "workload": name, "instances": n, "warps": int(rows.shape[0]), "solve_ms": solve_ms, "front_ms": front_ms,
            "solves_per_warp_mean": float(solves / rows.shape[0]), "adds_plus_drops_per_solve": float(changes / solves),
            "adds_mean": float(info[1].mean()), "drops_mean": float(info[2].mean()),
            "cycles_per_solve": float(busy / solves), "cycles_per_change_all_phases": float(busy / changes),
            "kernel_cycles_per_warp_max": float(kernel.max()), "kernel_cycles_per_warp_mean": float(kernel.mean()),
            "phases": {PHASES[k]: {"cycles_per_solve": float(tot[k] / solves), "share": float(tot[k] / busy)} for k in range(9)},
        })
        b.close()
    doc["sm_clock_mhz_reported"] = clock_mhz
    txt = json.dumps(doc, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
