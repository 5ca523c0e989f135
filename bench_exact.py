"""Exact QP mode (WBC_QP_EXACT), cold and warm-started (WBC_QP_WARM), against the default DENSE-AUL mode, timed alternately in
one process on one GPU.

For each workload three ctxs run the same device-resident control cycle, one per mode (default, exact, exact_warm), step by step
in turn: each step is timed with CUDA events on the launching stream with L2 flushed before it (bench.timed_device_loop).
Workloads:
  * frozen state -- standing_4096, trot_65536 and the 131 072-instance shard of mixed_terrain_1m, the seeded inputs of bench.py,
    repeated every step.  For exact_warm this is the warm start's best case: the previous cycle is this cycle.
  * moving state -- trot_rollout_4096 and trot_rollout_65536: cycle k of scenarios.trot_rollout at step k (warm-up steps
    included), the same cycle sequence for every mode's ctx, each ctx chaining its own observer state.
Per mode: solves/s, front and solve kernel ms (medians), the roofline of the solve kernel from the solver's own instrumented flop
count (qp_flops) against the measured DFMA peak, and the launch shape; for the exact modes the means over the timed steps of the
warm rows forced in (qp_info[6]), the GI loop's inequality additions, the drops and the share of instances warm-started; then how
many instances' torques differ between default and exact mode by more than 1e-6 relative, by contact mode.  The GPU's name and
power limit are read in the same run.  Prints one JSON document; --out also writes it to a file.

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

WORKLOADS = [("standing_4096", None), ("trot_65536", None), ("mixed_terrain_1m", 131072), ("trot_rollout_4096", 4096),
             ("trot_rollout_65536", 65536)]
MODES = (("default", False, False), ("exact", True, False), ("exact_warm", True, True))
FL_WARM_STARTED = 2048


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
    dev = env.dev
    rollout = name.startswith("trot_rollout")

    def to_dev(sc):
        return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    if rollout:
        n = per_gpu
        scs = [S.trot_rollout(n, k) for k in range(warmup + steps)]
        dev_ins = [to_dev(sc) for sc in scs]
        sc = scs[-1]
        obs0 = (np.zeros((6, n)), np.zeros((6, n)))
        res = {"workload": name, "instances": n, "state": "moving: cycle k of scenarios.trot_rollout(n, k) at step k (seed 5), "
               "the same cycle sequence on every mode's ctx, each chaining its own observer state from zero"}
    else:
        cfg = bench.workload_cfg(name)
        n_cfg = cfg.pop("n")
        n = per_gpu or n_cfg
        sc = S.make(n, **cfg)
        dev_ins = [to_dev(sc)] * (warmup + steps)
        obs0 = (sc["obs_yd"], sc["obs_yw"])
        res = {"workload": name, "instances": n, "mode_mix": cfg["mode_mix"], "terrain": cfg["terrain"], "pushes": cfg["pushes"],
               "seed": cfg["seed"], "state": "frozen: the same inputs every step (for exact_warm the warm start's best case: the "
               "previous cycle is this cycle)"}
    res.update({"steps": steps, "warmup": warmup, "l2": "flushed before every timed step (256 MiB write)"})
    legs = {}
    for mode, exact, warm in MODES:
        b = api.WbcBatch(max_batch=n, device=env.local_rank)
        b.set_observer_state(*obs0)
        out = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
               "status": torch.zeros(n, dtype=torch.int32, device=dev), "qp_info": torch.zeros(8, n, dtype=torch.int32, device=dev),
               "qp_flops": torch.zeros(n, dtype=torch.float64, device=dev)}
        legs[mode] = dict(batch=b, exact=exact, warm=warm, out=out, total=[], front=[], solve=[], forced=[], gi_adds=[], drops=[],
                          started=[])

    def stepper(leg, dev_in):
        def step(_):
            leg["batch"].cycle_device(dev_in, leg["out"], n, n, stream=env.sp, sync=False, exact=leg["exact"], warm=leg["warm"])
        return step

    for k in range(warmup):
        for leg in legs.values():
            stepper(leg, dev_ins[k])(0)
    torch.cuda.synchronize()
    for it in range(steps):                     # alternate the modes step by step
        for leg in legs.values():
            t, f, s_ = bench.timed_device_loop(env, leg["batch"], stepper(leg, dev_ins[warmup + it]), 1)
            leg["total"].append(t[0]); leg["front"].append(f[0]); leg["solve"].append(s_[0])
            if leg["exact"]:
                info = leg["out"]["qp_info"].cpu().numpy()
                leg["forced"].append(info[6].mean())
                leg["gi_adds"].append((info[1] - info[6] - (info[4] - info[3])).mean())
                leg["drops"].append(info[2].mean())
                leg["started"].append(((info[5] & FL_WARM_STARTED) != 0).mean())
    torch.cuda.synchronize()
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
            r["over_timed_steps"] = {"forced_additions_mean": float(np.mean(leg["forced"])),
                                     "gi_inequality_additions_mean": float(np.mean(leg["gi_adds"])),
                                     "drops_mean": float(np.mean(leg["drops"])), "warm_started_share": float(np.mean(leg["started"]))}
        res[mode] = r
    ta = legs["default"]["out"]["tau"].cpu().numpy().T
    tb = legs["exact"]["out"]["tau"].cpu().numpy().T
    rel = np.abs(ta - tb).max(axis=1) / np.maximum(1e-30, np.abs(tb).max(axis=1))
    res["tau_differs_1e-6_rel"] = {str(m): {"instances": int((sc["mode"] == m).sum()), "differ": int(((rel > 1e-6) & (sc["mode"] == m)).sum()),
                                             "worst_rel": float(rel[sc["mode"] == m].max()) if (sc["mode"] == m).any() else 0.0}
                                   for m in (0, 1, 2)}
    res["exact_over_default_solves_per_s"] = res["exact"]["solves_per_s"] / res["default"]["solves_per_s"]
    res["exact_warm_over_exact_solves_per_s"] = res["exact_warm"]["solves_per_s"] / res["exact"]["solves_per_s"]
    res["exact_warm_over_exact_solve_ms"] = res["exact_warm"]["solve_ms"] / res["exact"]["solve_ms"]
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
    doc = {"gpu": gpu_identity(), "library": os.environ.get("WBC_B200_LIB", "in-tree build"), "method": "three ctxs (one per mode) on the same seeded device-resident inputs, steps alternated; "
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
