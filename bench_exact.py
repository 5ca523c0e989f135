"""Exact QP mode (WBC_QP_EXACT) against the default DENSE-AUL mode, timed alternately in one process on one GPU.

For each workload (standing_4096, trot_65536 and the 131 072-instance shard of mixed_terrain_1m, the seeded inputs of bench.py)
two ctxs run the same device-resident control cycle, one per mode, step by step in turn: each step is timed with CUDA events on
the launching stream with L2 flushed before it (bench.timed_device_loop).  Per mode: solves/s, front and solve kernel ms
(medians), the roofline of the solve kernel from the solver's own instrumented flop count (qp_flops) against the measured DFMA
peak, and the launch shape; then how many instances' torques differ between the modes by more than 1e-6 relative, by contact
mode.  The GPU's name and power limit are read in the same run.  Prints one JSON document; --out also writes it to a file.

    python bench_exact.py [--steps K] [--warmup W] [--workloads a,b] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from wbc_quadruped_dob_b200 import scenarios as S  # noqa: E402

WORKLOADS = [("standing_4096", None), ("trot_65536", None), ("mixed_terrain_1m", 131072)]
MODES = (("default", False), ("exact", True))


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def run_workload(env, name, per_gpu, steps, warmup):
    import torch
    from wbc_quadruped_dob_b200 import api
    cfg = bench.workload_cfg(name)
    n_cfg = cfg.pop("n")
    n = per_gpu or n_cfg
    sc = S.make(n, **cfg)
    dev = env.dev
    dev_in = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    legs = {}
    for mode, exact in MODES:
        b = api.WbcBatch(max_batch=n, device=env.local_rank)
        b.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        out = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
               "status": torch.zeros(n, dtype=torch.int32, device=dev), "qp_info": torch.zeros(8, n, dtype=torch.int32, device=dev),
               "qp_flops": torch.zeros(n, dtype=torch.float64, device=dev)}
        legs[mode] = dict(batch=b, exact=exact, out=out, total=[], front=[], solve=[])

    def stepper(leg):
        def step(_):
            leg["batch"].cycle_device(dev_in, leg["out"], n, n, stream=env.sp, sync=False, exact=leg["exact"])
        return step

    for _ in range(warmup):
        for leg in legs.values():
            stepper(leg)(0)
    torch.cuda.synchronize()
    for it in range(steps):                     # alternate the modes step by step
        for leg in legs.values():
            t, f, s_ = bench.timed_device_loop(env, leg["batch"], stepper(leg), 1)
            leg["total"].append(t[0]); leg["front"].append(f[0]); leg["solve"].append(s_[0])
    torch.cuda.synchronize()
    res = {"workload": name, "instances": n, "mode_mix": cfg["mode_mix"], "terrain": cfg["terrain"], "pushes": cfg["pushes"],
           "seed": cfg["seed"], "steps": steps, "warmup": warmup, "l2": "flushed before every timed step (256 MiB write)"}
    peak = None
    for mode, leg in legs.items():
        b = leg["batch"]
        occ, smem, grid = b.solver_shape()
        kernel = b.last_solver_kernel
        if peak is None:
            peak = b.measure_dfma_peak()
        status = leg["out"]["status"].cpu().numpy()
        flops = leg["out"]["qp_flops"].cpu().numpy()
        info = leg["out"]["qp_info"].cpu().numpy()
        total, front, solve = (float(np.median(leg[k])) for k in ("total", "front", "solve"))
        r = {"solves_per_s": n / (total * 1e-3), "step_ms": total, "front_ms": front, "solve_ms": solve,
             "step_ms_min_max": [float(np.min(leg["total"])), float(np.max(leg["total"]))],
             "failed": int((status != 0).sum()),
             "solver_shape": {"kernel": kernel, "ctas_per_sm": occ, "smem_bytes": smem, "grid": grid},
             "flops_per_solve_mean": float(flops.mean()),
             "roofline": {"bound": "fp64", "flops_source": "the solver's own instrumented count (qp_flops)",
                          "achieved": float(flops.sum() / (solve * 1e-3)), "peak_measured_dfma": peak,
                          "frac": float(flops.sum() / (solve * 1e-3) / peak), "unit": "FLOP/s"}}
        if leg["exact"]:
            r["additions_mean"] = float(info[1].mean()); r["drops_mean"] = float(info[2].mean())
            r["drops_histogram"] = np.bincount(info[2]).tolist()
        res[mode] = r
    ta = legs["default"]["out"]["tau"].cpu().numpy().T
    tb = legs["exact"]["out"]["tau"].cpu().numpy().T
    rel = np.abs(ta - tb).max(axis=1) / np.maximum(1e-30, np.abs(tb).max(axis=1))
    res["tau_differs_1e-6_rel"] = {str(m): {"instances": int((sc["mode"] == m).sum()), "differ": int(((rel > 1e-6) & (sc["mode"] == m)).sum()),
                                             "worst_rel": float(rel[sc["mode"] == m].max()) if (sc["mode"] == m).any() else 0.0}
                                   for m in (0, 1, 2)}
    res["exact_over_default_solves_per_s"] = res["exact"]["solves_per_s"] / res["default"]["solves_per_s"]
    for leg in legs.values():
        leg["batch"].close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--workloads", default=",".join(w for w, _ in WORKLOADS), help="comma-separated subset of " + ", ".join(w for w, _ in WORKLOADS))
    args = ap.parse_args()
    pick = args.workloads.split(",")
    for w in pick:
        if w not in dict(WORKLOADS):
            raise SystemExit("unknown workload %r" % w)
    env = bench.Env(args)
    doc = {"gpu": gpu_identity(), "library": os.environ.get("WBC_B200_LIB", "in-tree build"), "method": "two ctxs (one per mode) on the same seeded device-resident inputs, steps alternated; "
           "medians of CUDA-event step times", "workloads": []}
    for name, per in [wl for wl in WORKLOADS if wl[0] in pick]:
        doc["workloads"].append(run_workload(env, name, per, args.steps, args.warmup))
    doc["gpu_after"] = gpu_identity()
    env.close()
    txt = json.dumps(doc, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
