"""bench.py's two rollout workloads (state that moves from cycle to cycle; see bench.py for the common contract).

trot_rollout   a herd of robots stepping through the trot gait with per-robot phase offsets (scenarios.trot_rollout): at every
               cycle ~2 % of the robots change contact mode, swing and stance solves are mixed, active sets drift.  The
               dispatch order of the solver's work queue is PREDICTED from each robot's previous cycle, so this is the
               workload that shows what that prediction is worth when the state moves: value (longest-first) beside
               value_fifo, and the rank correlation between predicted and actual solve cost.
push_sweep     BASELINE config 5: the 16 x 8 x 8 x 256 disturbance-rejection grid, closed loop through wbc_plant_step for
               400 cycles (1 s), observer rise time and steady-state error per gain reduced on the device and gathered with
               one NCCL all-reduce.
"""
import json
import os
import time

import numpy as np

from wbc_quadruped_dob_b200 import scenarios as S
from wbc_quadruped_dob_b200 import sharding

METRIC = "wbc_control_cycle_solves_per_sec"
UNIT = "solves/s"


def _spearman(a, b):
    ra = np.argsort(np.argsort(a)).astype(np.float64)
    rb = np.argsort(np.argsort(b)).astype(np.float64)
    ra -= ra.mean(); rb -= rb.mean()
    d = np.sqrt((ra * ra).sum() * (rb * rb).sum())
    return float((ra * rb).sum() / d) if d > 0 else 0.0


def bench_trot_rollout(env, args):
    import torch
    import bench as B
    from wbc_quadruped_dob_b200 import api
    rank, world, dev = env.rank, env.world, env.dev
    n = args.per_gpu or 4096
    steps, warmup = args.steps, args.warmup
    start = rank * n
    total_steps = warmup + steps
    # inputs of every cycle, staged in HBM once: the herd's state advances by pointing the cycle at the next slab
    host_sc = [S.trot_rollout(n, t, start=start) for t in range(total_steps)]
    dev_sc = [{k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items()} for sc in host_sc]
    batch = api.WbcBatch(max_batch=n, device=env.local_rank)
    dev_out = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev)}
    stat_out = dict(dev_out)
    stat_out.update(status=torch.zeros(n, dtype=torch.int32, device=dev), qp_info=torch.zeros(8, n, dtype=torch.int32, device=dev),
                    qp_flops=torch.zeros(n, dtype=torch.float64, device=dev))
    zero6 = np.zeros((6, n))
    sp = env.sp

    def run(fifo, outs_last=None):
        batch.fifo_dispatch = fifo
        batch.set_observer_state(zero6, zero6)
        for t in range(warmup):
            batch.cycle_device(dev_sc[t], dev_out, n, n, stream=sp, sync=False)
        torch.cuda.synchronize()
        env.barrier()
        ms, fr, so = B.timed_device_loop(env, batch, lambda it: batch.cycle_device(dev_sc[warmup + it], outs_last if (outs_last is not None and it == steps - 1) else dev_out,
                                                                                   n, n, stream=sp, sync=False), steps)
        env.barrier()
        return ms, fr, so

    sampler = B.ClockSampler(env.local_rank)
    sampler.start()
    t_wall0 = time.perf_counter()
    step_ms, front_ms, solve_ms = run(False, stat_out)
    t_wall = time.perf_counter() - t_wall0
    last = {k: stat_out[k].cpu().numpy() for k in dev_out} if args.dump_outputs and rank == 0 else None     # the fifo run overwrites them
    status = stat_out["status"].cpu().numpy()
    qp_info = stat_out["qp_info"].cpu().numpy()
    qp_flops = stat_out["qp_flops"].cpu().numpy()
    fifo_ms, _, _ = run(True)
    dfma_peak = batch.measure_dfma_peak()
    # ---- how good is the prediction?  actual cost of cycle t against the cost of cycle t-1 (what orders the queue), un-timed pass
    batch.fifo_dispatch = False
    batch.set_observer_state(zero6, zero6)
    prev, rho, flips = None, [], []
    for t in range(min(total_steps, 24)):
        batch.cycle_device(dev_sc[t], dev_out, n, n, stream=sp, sync=True)
        cyc = batch.last_solve_cycles(n).astype(np.float64)
        if prev is not None:
            rho.append(_spearman(prev, cyc))
            flips.append(float(np.mean(host_sc[t]["mode"] != host_sc[t - 1]["mode"])))
        prev = cyc
    # ---- e2e: host buffers through wbc_cycle, a fresh set of inputs every cycle
    pinned = [batch.pinned_inputs(sc) for sc in host_sc]
    out_pin = {"tau": batch.pinned((12, n)), "w": batch.pinned((6, n))}
    batch.set_observer_state(zero6, zero6)
    for t in range(warmup):
        batch.cycle(pinned[t], want=(), out=out_pin)
    env.barrier()
    t0 = time.perf_counter()
    for t in range(steps):
        out_host = batch.cycle(pinned[warmup + t], want=(), out=out_pin)
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    assert np.isfinite(out_host["tau"]).all()

    tot_ms, fifo_tot, e2e_s = env.max_over_ranks([float(step_ms.sum()), float(fifo_ms.sum()), e2e_s])
    stats = sharding.gather_stats(sharding.local_stats(n, status, qp_info, qp_flops, ms=tot_ms / steps), device=dev)
    line = None
    occ, smem, grid_ctas = batch.solver_shape()
    if rank == 0:
        total = n * world
        solve_avg = float(np.mean(solve_ms))
        achieved = float(qp_flops.sum()) / (solve_avg * 1e-3) / 1e12
        peak = dfma_peak / 1e12
        modes = np.bincount(host_sc[-1]["mode"], minlength=3) / float(n)
        line = {"metric": METRIC, "value": total * steps / (tot_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": tot_ms / steps, "p50_ms": float(np.median(step_ms)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "trot_rollout: %d robots per GPU x %d GPU(s) trotting with per-robot phase offsets (stance, swing{BR,FL}, stance, swing{BL,FR}; "
                                       "46 cycles each), observer chained, inputs of every cycle resident in HBM; mode mix at the last cycle %s" % (n, world, np.round(modes, 3).tolist()),
                           "instances_per_gpu": n, "global_batch": total, "parallelism": "shard%d" % world, "l2": "flushed between timed steps (256 MiB write)",
                           "dispatch": "longest-first, predicted from each robot's PREVIOUS cycle (state and contact mode have moved since)",
                           "solver_launch": "%d persistent one-warp CTAs (%d per SM), %d B shared memory each" % (grid_ctas, occ, smem)},
                "clocks": clocks,
                "value_fifo": total * steps / (fifo_tot * 1e-3),
                "dispatch_gain": fifo_tot / tot_ms,
                "dispatch_prediction": {"spearman_prev_vs_actual_cost": {"mean": float(np.mean(rho)), "min": float(np.min(rho)), "cycles": len(rho)},
                                        "robots_changing_mode_per_cycle": float(np.mean(flips))},
                "e2e": {"value": total * steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n * B.IN_BYTES, "d2h_bytes_per_step": n * B.OUT_BYTES},
                "gpu_launches": 2 * steps, "e2e_gpu_launches": 2 * steps,
                "roofline": {"bound": "fp64", "kernel": batch.last_solver_kernel,
                             "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                             "algorithmic_bytes_per_launch": B.algorithmic_bytes(host_sc[-1]["mode"], False),
                             "flops_per_solve": float(qp_flops.mean()), "kernel_ms": solve_avg, "front_kernel_ms": float(np.mean(front_ms)),
                             "peak_source": "own DFMA microbenchmark in this process (MEASURED_PEAKS.json has no FP64 figure)"},
                "stats": {"solver_failures": stats["solver_failures"], "mean_ncholesky": stats["sum_ncholesky"] / total,
                          "mean_outer_its": stats["sum_outer_its"] / total, "max_kkt_dim": stats["max_kkt_dim"], "wall_s_timed_region": t_wall}}
        if not args.no_cpu_baseline and world == 1 and not B.reference_built():
            line["cpu_baseline"] = B.NO_CPU_BASELINE
        elif not args.no_cpu_baseline and world == 1:
            kind, tot, _ = B.cpu_reference_run(dict(host_sc[-1], obs_yd=zero6, obs_yw=zero6), 1, 0, min(n, 4096), env.cores)
            line["cpu_baseline"] = {"value": min(n, 4096) / tot, "unit": UNIT, "cores": env.cores, "kind": kind,
                                    "sample": "one pass over the first %d robots at the last cycle, all %d host threads" % (min(n, 4096), env.cores)}
        if last is not None:
            B.dump_outputs(args.dump_outputs, last)
    batch.close()
    return line


def bench_push_sweep(env, args):
    """Config 5 as SURVEY.md 8(d) row 5 states it: 262 144 instances (16 directions x 8 magnitudes x 8 observer gains x 256 states)
    sharded over the ranks (strong scaling), 400 closed-loop cycles = 1 s, everything resident in HBM; per observer gain the
    rise time of the estimate (first cycle at which its projection on the true push reaches 90 %) and the steady-state error
    (mean relative error over the last 40 cycles), reduced on the device, one NCCL all-reduce."""
    import torch
    import torch.distributed as dist
    import bench as B
    from wbc_quadruped_dob_b200 import api
    rank, world, dev = env.rank, env.world, env.dev
    total = B.SWEEP_TOTAL if args.per_gpu is None else args.per_gpu * world
    lo, hi = sharding.shard_range(total, rank, world)
    n = hi - lo
    cycles = args.steps                    # --steps or --sweep-cycles, 400 = 1 s by default
    dyn_plant = getattr(args, "plant", "momentum") == "dynamics"
    tail = max(1, min(40, cycles // 4))
    sc = S.push_sweep(n=n, start=lo)
    sc.pop("grid", None)
    if getattr(args, "plant", "momentum") == "dynamics":
        # the articulated robot really moves: hold the pose it starts in (the momentum plant keeps joints and orientation frozen, so
        # there the scenario's desired CoM offset only loads the QP)
        com0, _ = S.forward_kinematics(sc["base_pos"], sc["base_rot"], sc["q"])
        sc["com_des_pos"] = np.vstack([com0.T, sc["base_rpy"]])
    batch = api.WbcBatch(max_batch=n, device=env.local_rank)
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    din = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dout = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev),
            "x": torch.zeros(30, n, dtype=torch.float64, device=dev)}
    sout = dict(dout)
    sout.update(status=torch.zeros(n, dtype=torch.int32, device=dev), qp_info=torch.zeros(8, n, dtype=torch.int32, device=dev),
                qp_flops=torch.zeros(n, dtype=torch.float64, device=dev))
    push = din["push"]
    pscale = push.abs().amax(dim=0)
    pnorm2 = (push[:3] * push[:3]).sum(dim=0)
    gains = torch.tensor(S.SWEEP_GAINS, dtype=torch.float64, device=dev)
    gidx = torch.bucketize(din["obs_gain"], gains)                       # gain index of every instance
    rise = torch.full((n,), -1, dtype=torch.int64, device=dev)
    ss_acc = torch.zeros(n, dtype=torch.float64, device=dev)
    fail = torch.zeros((), dtype=torch.int64, device=dev)
    sp = env.sp
    sampler = B.ClockSampler(env.local_rank)
    sampler.start()
    env.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(cycles)]
    for c in range(cycles):
        outs = sout if c == cycles - 1 else dout
        ev[c][0].record(env.stream)
        batch.cycle_device(din, outs, n, n, stream=sp, sync=False)
        if dyn_plant:
            # SURVEY.md 8f-2: the articulated robot on rigid contacts under the commanded torques and the push
            batch.plant_dynamics_step(din, outs["tau"], din["push"], n=n, ld=n, substeps=5, gamma=100.0, stream=sp, sync=False)
        else:
            batch.plant_step(din["base_pos"], din["base_vel"], din["push"], foot_force=din["foot_force"], x=outs["x"], n=n, ld=n, stream=sp, sync=False)
        ev[c][1].record(env.stream)
        # metrics of this cycle, on the device, outside the timed bracket
        w = dout["w"]
        proj = (w[:3] * push[:3]).sum(dim=0) / pnorm2
        rise = torch.where((rise < 0) & (proj >= 0.9), torch.full_like(rise, c + 1), rise)
        if c >= cycles - tail:
            ss_acc += (w - push).abs().amax(dim=0) / pscale
    torch.cuda.synchronize()
    env.barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    tot_ms = float(step_ms.sum())
    status = sout["status"].cpu().numpy()
    qp_info = sout["qp_info"].cpu().numpy()
    qp_flops = sout["qp_flops"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        B.dump_outputs(args.dump_outputs, {k: sout[k].cpu().numpy() for k in dout})
    # ---- per-gain reduction on the device, then ONE all-reduce of the packed vector (sums) and one of the maxima
    G = len(S.SWEEP_GAINS)
    ss = ss_acc / tail
    never = (rise < 0)
    rise_f = torch.where(never, torch.full_like(rise, cycles), rise).to(torch.float64)
    cnt = torch.bincount(gidx, minlength=G).to(torch.float64)
    sums = torch.cat([cnt, torch.bincount(gidx, weights=rise_f, minlength=G), torch.bincount(gidx, weights=ss, minlength=G),
                      torch.bincount(gidx, weights=never.to(torch.float64), minlength=G)])
    maxs = torch.stack([torch.zeros(G, dtype=torch.float64, device=dev).scatter_reduce(0, gidx, rise_f, reduce="amax"),
                        torch.zeros(G, dtype=torch.float64, device=dev).scatter_reduce(0, gidx, ss, reduce="amax")]).reshape(-1)
    maxs = torch.cat([maxs, torch.tensor([tot_ms, din["base_vel"][:3].abs().max().item()], dtype=torch.float64, device=dev)])
    if world > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        dist.all_reduce(maxs, op=dist.ReduceOp.MAX)
    sums, maxs = sums.cpu().numpy(), maxs.cpu().numpy()
    tot_ms = float(maxs[2 * G])
    stats = sharding.gather_stats(sharding.local_stats(n, status, qp_info, qp_flops, ms=tot_ms / cycles), device=dev)
    solve_ms = batch.last_timing()[1]          # before the peak measurement, which reuses the ctx's events
    dfma_peak = batch.measure_dfma_peak()
    occ, smem, grid_ctas = batch.solver_shape()
    line = None
    if rank == 0:
        cnt = sums[0:G]
        per_gain = {}
        for g, k in enumerate(S.SWEEP_GAINS):
            per_gain[str(k)] = {"instances": int(cnt[g]), "rise_time_s_mean": 0.0025 * sums[G + g] / cnt[g], "rise_time_s_max": 0.0025 * maxs[g],
                                "never_rose": int(sums[3 * G + g]), "steady_state_rel_err_mean": sums[2 * G + g] / cnt[g], "steady_state_rel_err_max": maxs[G + g],
                                "first_order_prediction": {"rise_time_s": float(np.log(10.0) * (1.0 / k + 0.0025)), "rel_err_at_end": float((1.0 + k * 0.0025) ** (-cycles))}}
        achieved = float(qp_flops.sum()) / (solve_ms * 1e-3) / 1e12
        line = {"metric": METRIC, "value": total * cycles / (tot_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": cycles, "warmup": 0,
                "ms_per_step": tot_ms / cycles, "p50_ms": float(np.median(step_ms)), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "push_sweep: %d instances (16 push directions x 8 magnitudes 5..80 N x 8 observer gains x 256 states) over %d GPU(s), "
                                       "%d closed-loop cycles (%.2f s) through %s, everything resident in HBM" % (total, world, cycles, cycles * 0.0025,
                                                                                                                              "wbc_plant_dynamics_step (forward dynamics, rigid contacts, 5 substeps)" if dyn_plant else "wbc_plant_step"),
                           "instances_per_gpu": n, "global_batch": total, "parallelism": "shard%d" % world, "l2": "not flushed (a rollout keeps its state warm)",
                           "scaling_note": "fixed grid sharded over the ranks (strong scaling); one step = one closed-loop cycle of every instance",
                           "solver_launch": "%d persistent one-warp CTAs (%d per SM), %d B shared memory each" % (grid_ctas, occ, smem)},
                "clocks": clocks,
                "e2e": {"value": total * cycles / wall, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "note": "a closed-loop rollout has no per-cycle host traffic: the plant runs on the device; wall clock of the whole rollout including the per-cycle metric reductions"},
                "gpu_launches": 3 * cycles,
                "roofline": {"bound": "fp64", "kernel": batch.last_solver_kernel,
                             "achieved": achieved, "peak": dfma_peak / 1e12, "unit": "TFLOP/s", "frac": achieved / (dfma_peak / 1e12), "traffic": None,
                             "kernel_ms": float(solve_ms), "flops_per_solve": float(qp_flops.mean())},
                "stats": {"solver_failures": stats["solver_failures"], "mean_ncholesky": stats["sum_ncholesky"] / total, "wall_s_timed_region": wall,
                          "sweep": {"cycles": cycles, "sim_time_s": cycles * 0.0025, "steady_state_window_cycles": tail, "per_gain": per_gain,
                                    "max_abs_base_lin_vel": float(maxs[2 * G + 1])}}}
    batch.close()
    return line
