#!/usr/bin/env python3
"""bench.py -- WBC control-cycle solves/s on N B200s (one process per GPU), see DESIGN.md "Measurement".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = one full control cycle (update -> Fgrf -> estimate -> QP assembly -> DENSE-AUL solve -> tau) over one
batch of synthetic DogBot instances.  At N=1 the workload is BASELINE.json configs[1] (4096 standing instances);
with N ranks every rank runs its own shard of N x that batch (weak scaling, no data-path collective; one NCCL
all-reduce of a 7-double statistics vector at the end).

  value     solves/s, inputs and outputs resident in HBM (device pointers through the C ABI), CUDA-event timed
  e2e       solves/s through the reference-facing call with HOST buffers: H2D + kernels + D2H inside the timed region
  roofline  the solve kernel: instrumented algorithmic FP64 flops / CUDA-event time vs the DFMA peak measured in
            the same process; HBM figures beside it (the path is FP64-pipe/latency bound, not HBM bound)
  cpu_baseline  the CPU oracle (C restatement + the reference's own ALGLIB) on all host cores, same inputs

`--impl reference` times that CPU path alone (rank 0 only).  Where the reference's ALGLIB is not built, the B200 arm reports
cpu_baseline as unavailable and `--impl reference` fails.

`--dump-outputs DIR` writes what the timed loop computed in its last step (rank 0's shard), one DIR/<name>.npy per output the
caller receives, so that two builds can be compared output for output: the inputs are seeded, the same arguments give the same ones.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from wbc_quadruped_dob_b200 import scenarios as S           # noqa: E402
from wbc_quadruped_dob_b200 import sharding                 # noqa: E402

METRIC = "wbc_control_cycle_solves_per_sec"
UNIT = "solves/s"
FRONT_FLOPS = 32.0e3      # dynamics + CoM transform + observer + assembly per instance (SURVEY.md 8d)
IN_BYTES = 8 * 93 + 4     # algorithmic input bytes per instance (flat ground)
OUT_BYTES = 8 * 18        # tau + w


REPLAY = "trot_replay_single"  # BASELINE config 1: ONE robot replaying a 184-cycle synthetic trot, one control cycle per step (latency case)
SWEEP = "push_sweep"          # BASELINE config 5: closed-loop disturbance-rejection sweep, fixed 262144-instance grid
ROLLOUT = "trot_rollout"      # evolving-state herd: every robot steps through the trot gait, modes and active sets change from cycle to cycle
QPREC_DOUBLES = 576           # front kernel -> solver record (wbc_types.h)
SWEEP_TOTAL = S.SWEEP_DIRECTIONS * len(S.SWEEP_MAGNITUDES) * len(S.SWEEP_GAINS) * S.SWEEP_STATES


def workload_cfg(name):
    if name == SWEEP:
        return dict(n=SWEEP_TOTAL, mode_mix=(1.0, 0.0, 0.0), pushes="grid 16 directions x 8 magnitudes (5..80 N)", terrain=False, seed=4)
    cfg = dict(S.CONFIGS[name])
    return cfg


def cpu_reference_run(sc, steps, warmup, sample, cores):
    """The reference's CPU path: oracle restatement of main.cpp's cycle + the reference's own ALGLIB (oracle/_ref)."""
    from oracle import oracle_py as op
    op.build(ref=True)
    kind = "reference" if op.have_ref() else "port"
    if not op.have_ref():
        raise SystemExit("oracle/_ref/libref_alglib_qp.so is missing: build it where /root/reference exists")
    sub = {k: (np.ascontiguousarray(v[..., :sample]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    times = []
    for it in range(warmup + steps):
        _, secs = op.run_cycle_batch(sub, nthreads=cores)
        if it >= warmup:
            times.append(secs)
    return kind, float(np.sum(times)), times


def reference_built():
    from oracle import oracle_py as op
    op.build(ref=True)
    return op.have_ref()


NO_CPU_BASELINE = {"value": None, "unit": UNIT, "kind": "unavailable",
                   "note": "the reference's ALGLIB (oracle/_ref/libref_alglib_qp.so) is not built, so the CPU path cannot run"}
DUMP_LIMIT = 64_000_000            # bytes on disk, all files of one dump together
NPY_HEADER_MAX = 1024               # room left per .npy file for its header (numpy writes 128 bytes for these shapes)


def dump_outputs(path, arrays):
    """--dump-outputs: each [k, n] output as path/<name>.npy in float64.  Above DUMP_LIMIT bytes on disk in all, the same fixed, seeded
    sample of instances (columns) is taken from every output, and the sampled instance indices are written as instances.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[-1]
    per_instance = sum(a.nbytes // n for a in arrays.values())
    if per_instance * n + NPY_HEADER_MAX * len(arrays) > DUMP_LIMIT:
        room = DUMP_LIMIT - NPY_HEADER_MAX * (len(arrays) + 1)
        keep = np.sort(np.random.default_rng(0).choice(n, room // (per_instance + 8), replace=False))
        arrays = {k: a[..., keep] for k, a in arrays.items()}
        arrays["instances"] = keep.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a))


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML, else nvidia-smi)."""

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    def run(self):
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self.samples.append(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
                    try:
                        r = self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, nm in names.items():
                        if r & bit and nm != "gpu_idle":
                            self.reasons.add(nm)
                else:
                    import subprocess
                    o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                        "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    a, b = o.strip().split(",")
                    self.samples.append(int(a)); self.max_mhz = int(b)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def single_robot_replay(args):
    """BASELINE configs[0]: one DogBot, one control cycle per step (the 400 Hz loop of main.cpp:836-1955), observer state
    chained on the device.  Reports cycles/s (= solves/s), p50/p95 latency of a cycle, device-resident and end to end,
    beside the CPU oracle + reference ALGLIB running the same replay on one host thread."""
    import torch
    from wbc_quadruped_dob_b200 import api
    sc = S.trot_replay()
    ncyc = sc["mode"].shape[0]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    batch = api.WbcBatch(max_batch=1, device=0)
    dev_in = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray) and k not in ("obs_yd", "obs_yw")}
    dev_out = {"tau": torch.zeros(12, 1, dtype=torch.float64, device=dev), "w": torch.zeros(6, 1, dtype=torch.float64, device=dev)}
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream

    def dev_cycle(i):
        one = {k: (v[i:] if v.dim() == 1 else v[:, i:]) for k, v in dev_in.items()}     # pointer offset, ld = ncyc
        batch.cycle_device(one, dev_out, 1, ncyc, stream=sp, sync=False)

    host = [{k: (np.ascontiguousarray(v[..., i:i + 1]) if isinstance(v, np.ndarray) else v) for k, v in sc.items()} for i in range(ncyc)]
    steps, warm = (ncyc if args.steps is None else args.steps), args.warmup
    batch.set_observer_state(np.zeros((6, 1)), np.zeros((6, 1)))
    for i in range(warm):
        dev_cycle(i % ncyc)
    torch.cuda.synchronize()
    batch.set_observer_state(np.zeros((6, 1)), np.zeros((6, 1)))
    sampler = ClockSampler(0)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for it in range(steps):
        ev[it][0].record(stream)
        dev_cycle(it % ncyc)
        ev[it][1].record(stream)
        ev[it][1].synchronize()
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    last = {k: v.cpu().numpy() for k, v in dev_out.items()}
    batch.set_observer_state(np.zeros((6, 1)), np.zeros((6, 1)))
    e2e_ms = []
    for it in range(warm + steps):
        t0 = time.perf_counter()
        out = batch.cycle(host[it % ncyc], want=())
        if it >= warm:
            e2e_ms.append(1e3 * (time.perf_counter() - t0))
    clocks = sampler.stop()
    e2e_ms = np.array(e2e_ms)
    line = {"metric": METRIC, "value": 1e3 / float(step_ms.mean()), "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": warm,
            "ms_per_step": float(step_ms.mean()), "p50_ms": float(np.median(step_ms)), "p95_ms": float(np.percentile(step_ms, 95)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s: ONE DogBot, 184-cycle synthetic trot replay (46 stance + 46 swing{BR,FL} + 46 stance + 46 swing{BL,FR}), one control cycle per step, observer chained; timed: the first %d cycles of the replay (wrapping)" % (REPLAY, steps),
                       "instances_per_gpu": 1, "global_batch": 1, "parallelism": "single robot", "l2": "not flushed (a 400 Hz loop keeps its working set warm)"},
            "clocks": clocks,
            "e2e": {"value": 1e3 / float(e2e_ms.mean()), "unit": UNIT, "p50_ms": float(np.median(e2e_ms)), "p95_ms": float(np.percentile(e2e_ms, 95)),
                    "h2d_bytes_per_step": IN_BYTES, "d2h_bytes_per_step": OUT_BYTES},
            "gpu_launches": 2 * steps}
    if not args.no_cpu_baseline and not reference_built():
        line["cpu_baseline"] = NO_CPU_BASELINE
    elif not args.no_cpu_baseline:
        from oracle import oracle_py as op
        t0 = time.perf_counter()
        yd, yw = np.zeros((6, 1)), np.zeros((6, 1))
        for i in range(steps):
            one = dict(host[i % ncyc]); one["obs_yd"], one["obs_yw"] = yd, yw
            ref, _ = op.run_cycle_batch(one, nthreads=1)
            yd, yw = ref["yd"].T.copy(), ref["yw"].T.copy()
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": steps / dt, "unit": UNIT, "cores": 1, "kind": "reference" if op.have_ref() else "port",
                                "sample": "the same %d timed cycles of the %d-cycle replay, one host thread (the reference's control loop is single-threaded), %.3f ms per cycle"
                                          % (steps, ncyc, 1e3 * dt / steps)}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    print(json.dumps(line))
    batch.close()
    return 0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 30; the whole %s, 184 cycles; for %s 400 closed-loop cycles = 1 s)" % (REPLAY, SWEEP))
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="standing_4096", choices=sorted(S.CONFIGS) + [SWEEP, REPLAY, ROLLOUT])
    ap.add_argument("--per-gpu", type=int, default=None, help="instances per GPU (default: the workload's own size, 1M config: /8)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="headline workload only: skip the `also` lines (trot_65536, mixed_terrain_1m shard) and value_fifo")
    ap.add_argument("--traj-on-device", action="store_true",
                    help="e2e loop only: the plan's spline tables live in HBM and are sampled on the GPU each step (SURVEY 8f-1); "
                         "the 36 desired-trajectory doubles per instance are not sent from the host")
    ap.add_argument("--fifo", action="store_true", help="index-order work queue (WBC_FIFO_DISPATCH) instead of longest-first")
    ap.add_argument("--plant", default="momentum", choices=["momentum", "dynamics"],
                    help="push_sweep: the plant that closes the loop -- the CoM-momentum integrator of SURVEY 8d row 5 (default) or forward dynamics with rigid contacts (SURVEY 8f-2)")
    ap.add_argument("--sweep-cycles", type=int, default=None, help="push_sweep: closed-loop cycles of the rollout, another name for --steps there")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy, float64, at most 64 MiB (a seeded sample of instances beyond)")
    args = ap.parse_args()
    if args.workload == SWEEP and args.impl == "b200":
        if None not in (args.steps, args.sweep_cycles) and args.steps != args.sweep_cycles:
            ap.error("--steps and --sweep-cycles both set the push_sweep's timed cycles and disagree")
        args.steps = args.sweep_cycles = next(v for v in (args.steps, args.sweep_cycles, 400) if v is not None)
    elif args.steps is None and args.workload != REPLAY:       # the replay's default is its length, set where it is loaded
        args.steps = 30
    args.warmup = max(args.warmup, 3)
    return args


def algorithmic_bytes(mode, terrain):
    """SURVEY.md 8(d): 1024 B per solve (97 doubles in, 31 out), +144 B for a swing solve (18 swing-foot reference doubles are
    only read then), +320 B with per-foot terrain frames (40 doubles)."""
    n = int(mode.shape[0])
    return n * 1024 + int(np.count_nonzero(mode != 0)) * 144 + (n * 320 if terrain else 0)


class Env:
    """One rank's CUDA context for the run: device, the stream every launch and event goes to, the process group."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200: the CUDA path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.dev = torch.device("cuda", self.local_rank)
        # a dedicated non-default stream: the C ABI treats a NULL stream as "use the ctx's own stream", and
        # torch.cuda.Event only sees work on the stream it is recorded on -- kernels, L2 flush and events share this one
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        self.sp = self.stream.cuda_stream
        assert self.sp != 0
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)
        self.cores = os.cpu_count() or 1

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_device_loop(env, batch, step, steps, flush=True):
    """K device-resident steps, one CUDA-event pair per step on the launching stream; L2 flushed between steps."""
    torch = env.torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    solve_ms, front_ms = [], []
    for it in range(steps):
        if flush:
            env.flush.fill_(it & 0xFF)             # evict L2 between timed steps
        ev[it][0].record(env.stream)
        step(it)
        ev[it][1].record(env.stream)
        f, s_ = batch.last_timing()                # waits for this step's last event
        front_ms.append(f); solve_ms.append(s_)
    torch.cuda.synchronize()
    return np.array([a.elapsed_time(b) for a, b in ev]), np.array(front_ms), np.array(solve_ms)


def bench_batch(env, args, name, steps, warmup, per_gpu=None, cpu_baseline=False, fifo_steps=0, fifo=False, traj_on_device=False, dump=None):
    """One workload on this rank's shard: device-resident loop (`value`), end-to-end loop through wbc_cycle with host buffers
    (`e2e`), roofline of the solve kernel, statistics gathered over the ranks.  Returns the JSON line (rank 0) or None.
    dump: directory for the device-resident loop's last outputs (dump_outputs)."""
    import torch
    from wbc_quadruped_dob_b200 import api
    rank, world, dev = env.rank, env.world, env.dev
    cfg = workload_cfg(name)
    n_cfg = cfg.pop("n")
    sweep = name == SWEEP
    per_gpu = per_gpu or (n_cfg // 8 if name == "mixed_terrain_1m" else (n_cfg // world if sweep else n_cfg))
    config = {"workload": "%s: %d DogBot instances per GPU x %d GPU(s), 18-DoF, mode mix %s, pushes=%s, terrain=%s, seed %d" % (
        name, per_gpu, world, cfg["mode_mix"], cfg["pushes"], cfg["terrain"], cfg["seed"]),
        "instances_per_gpu": per_gpu, "global_batch": per_gpu * world, "parallelism": "shard%d" % world,
        "l2": "flushed between timed steps (256 MiB write)",
        "dispatch": "fifo" if fifo else "longest-first, predicted from each instance's previous cycle (results are order-independent)",
        "solver": "DENSE-AUL/QQP restatement, reference settings (1e-2, 1e4, 5)"}
    lo, hi = sharding.shard_range(per_gpu * world, rank, world)
    n = hi - lo
    sc = S.push_sweep(n=n, start=lo) if sweep else S.make(n, start=lo, **cfg)
    sc.pop("grid", None)
    batch = api.WbcBatch(max_batch=n, device=env.local_rank)
    batch.fifo_dispatch = fifo
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    dev_in = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in sc.items() if isinstance(v, np.ndarray)}
    dev_out = {"tau": torch.zeros(12, n, dtype=torch.float64, device=dev), "w": torch.zeros(6, n, dtype=torch.float64, device=dev)}
    stat_out = dict(dev_out)
    stat_out.update(status=torch.zeros(n, dtype=torch.int32, device=dev), qp_info=torch.zeros(8, n, dtype=torch.int32, device=dev),
                    qp_flops=torch.zeros(n, dtype=torch.float64, device=dev))
    sp = env.sp
    if sweep:
        # closed loop: the plant needs the commanded forces x[18:30] every cycle; observer gain per instance
        dev_out["x"] = torch.zeros(30, n, dtype=torch.float64, device=dev)
        stat_out["x"] = dev_out["x"]
        config["scaling_note"] = "fixed grid of %d instances sharded over the ranks (strong scaling); one step = one closed-loop cycle" % SWEEP_TOTAL

    def step(outs):
        batch.cycle_device(dev_in, outs, n, n, stream=sp, sync=False)
        if sweep:
            batch.plant_step(dev_in["base_pos"], dev_in["base_vel"], dev_in["push"], foot_force=dev_in["foot_force"], x=outs["x"], n=n, ld=n,
                             stream=sp, sync=False)

    for it in range(warmup):
        step(stat_out if it == warmup - 1 else dev_out)
    torch.cuda.synchronize()
    occ, smem, grid_ctas = batch.solver_shape()
    config["solver_launch"] = "%d persistent one-warp CTAs (up to %d resident per SM; %d B of shared memory per solve), %s" % (
        grid_ctas, occ, smem, "stage tasks with SM roles" if batch.last_solver_kernel == "wbc_solve_staged_kernel" else "one warp per solve")
    status = stat_out["status"].cpu().numpy()
    qp_info = stat_out["qp_info"].cpu().numpy()
    qp_flops = stat_out["qp_flops"].cpu().numpy()
    dfma_peak = batch.measure_dfma_peak()

    # ---- timed region: K steps, device-resident
    sampler = ClockSampler(env.local_rank)
    sampler.start()
    env.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    step_ms, front_ms, solve_ms = timed_device_loop(env, batch, lambda it: step(dev_out), steps)
    env.barrier()
    t_wall = time.perf_counter() - t_wall0
    last = {k: v.cpu().numpy() for k, v in dev_out.items()} if dump and rank == 0 else None     # the loops below overwrite dev_out
    tot_ms = float(step_ms.sum())
    launches = (3 if sweep else 2) * steps
    sweep_stats = None
    if sweep:
        # how far the observer got after warmup + steps closed-loop cycles, per gain (rank 0's shard)
        w_now = dev_out["w"].cpu().numpy()
        rel = np.abs(w_now - sc["push"]).max(axis=0) / np.abs(sc["push"]).max(axis=0)
        sweep_stats = {"cycles": warmup + steps, "sim_time_s": (warmup + steps) * 0.0025,
                       "w_rel_err_by_gain": {str(g): float(rel[sc["obs_gain"] == g].max()) for g in np.unique(sc["obs_gain"])},
                       "max_abs_base_lin_vel": float(dev_in["base_vel"][:3].abs().max().item())}

    # ---- the same loop with index-order dispatch (how much the longest-first order is worth on this workload)
    fifo_ms = None
    if fifo_steps > 0 and not fifo and not sweep:
        batch.fifo_dispatch = True
        batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
        for it in range(warmup):
            step(dev_out)
        torch.cuda.synchronize()
        fm, _, _ = timed_device_loop(env, batch, lambda it: step(dev_out), fifo_steps)
        fifo_ms = float(fm.sum()) / fifo_steps
        batch.fifo_dispatch = False

    # ---- e2e: host buffers through the C ABI (H2D + kernels + D2H inside the timed region)
    e2e_steps = steps
    want = ("x",) if sweep else ()
    # the caller's arrays live in page-locked host memory (wbc_host_alloc), as a controller process feeding the
    # batch every cycle would keep them: wbc_cycle then DMAs them directly (pageable arrays take its bounce buffer)
    sc_host = batch.pinned_inputs(sc)
    for k in ("push",):
        if k in sc_host and isinstance(sc_host[k], np.ndarray):
            sc_host[k] = batch.pinned_copy(np.ascontiguousarray(sc_host[k]))
    out_pin = {"tau": batch.pinned((12, n)), "w": batch.pinned((6, n))}
    if sweep:
        out_pin["x"] = batch.pinned((30, n))
    traj = None
    if traj_on_device and not sweep:
        # a plan whose splines start at the scenario's desired pose; sampled at t = 0 it reproduces the workload's inputs
        traj = S.make_trajectory(sc, nseg=3, seed=11, match_acc=True)
        batch.set_trajectory(traj)
        sc_host = batch.pinned_inputs({k: v for k, v in sc.items() if k not in api.TRAJ_FIELDS})
        config["trajectory"] = "sampled on the device every step from per-instance spline tables (3 polynomials per spline) at t = 0"

    def e2e_step():
        if traj is not None:
            batch.sample_trajectory(n, t_all=0.0)
            return batch.cycle(sc_host, want=want, out=out_pin, sampled_traj=True)
        out = batch.cycle(sc_host, want=want, out=out_pin)
        if sweep:   # host-side rollout: the plant's H2D/D2H copies are part of the step too
            batch.plant_step(sc_host["base_pos"], sc_host["base_vel"], sc_host["push"], foot_force=sc_host["foot_force"], x=out["x"])
        return out
    # same observer trajectory as the device-resident loop: the estimate feeds back into the QP (main.cpp:1032), so the
    # work per cycle drifts as the observer integrates; both loops start from the scenario's initial observer state
    batch.set_observer_state(sc["obs_yd"], sc["obs_yw"])
    for _ in range(warmup):
        e2e_step()
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out_host = e2e_step()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    assert np.isfinite(out_host["tau"]).all()

    # ---- max over ranks, statistics gather (the only collective)
    tot_ms, e2e_s = env.max_over_ranks([tot_ms, e2e_s])
    if fifo_ms is not None:
        fifo_ms = env.max_over_ranks([fifo_ms])[0]
    stats = sharding.gather_stats(sharding.local_stats(n, status, qp_info, qp_flops, ms=tot_ms / steps), device=dev)
    total_inst = per_gpu * world
    value = total_inst * steps / (tot_ms * 1e-3)
    e2e_val = total_inst * e2e_steps / e2e_s
    line = None
    if rank == 0:
        solve_avg_ms = float(np.mean(solve_ms))
        flops_launch = float(qp_flops.sum())
        achieved = flops_launch / (solve_avg_ms * 1e-3) / 1e12
        peak = dfma_peak / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        alg_bytes = algorithmic_bytes(sc["mode"], sc.get("terrain") is not None)
        hbm_ach = alg_bytes / (float(np.mean(step_ms)) * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(name)
            if tr and per_gpu == n_cfg:
                traffic, traffic_src = tr["bytes_per_launch"], tr["source"]
        except Exception:
            pass
        roofline = {"bound": "fp64", "kernel": batch.last_solver_kernel,
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)", "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "algorithmic_bytes_note": "SURVEY 8(d): 1024 B per solve, +144 B per swing solve, +320 B with terrain frames",
                    "intermediate_bytes_per_launch": n * 8 * QPREC_DOUBLES,
                    "intermediate_note": "front kernel -> solver QP record (%d doubles per solve), written once and read once; not algorithmic traffic" % QPREC_DOUBLES,
                    "peak_source": "own DFMA microbenchmark in this process (MEASURED_PEAKS.json has no FP64 figure)",
                    "flops_per_solve": flops_launch / n, "kernel_ms": solve_avg_ms, "front_kernel_ms": float(np.mean(front_ms)),
                    "resident_solver_warps_per_sm": occ,
                    "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": tot_ms / steps, "p50_ms": float(np.median(step_ms)), "higher_is_better": True, "scaling": "strong" if sweep else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": n * (IN_BYTES - (36 * 8 if traj_on_device and not sweep else 0) + (8 + 57 * 8 if sweep else 0)),
                        "d2h_bytes_per_step": n * (OUT_BYTES + (30 * 8 + 21 * 8 if sweep else 0))},
                "gpu_launches": launches, "e2e_gpu_launches": (3 if (sweep or (traj_on_device and not sweep)) else 2) * e2e_steps, "roofline": roofline,
                "stats": {"solver_failures": stats["solver_failures"], "mean_ncholesky": stats["sum_ncholesky"] / total_inst,
                          "mean_outer_its": stats["sum_outer_its"] / total_inst, "max_kkt_dim": stats["max_kkt_dim"],
                          "wall_s_timed_region": t_wall}}
        if fifo_ms is not None:
            line["value_fifo"] = total_inst / (fifo_ms * 1e-3)
            line["dispatch_gain"] = line["value"] / line["value_fifo"]
            line["value_fifo_note"] = "same workload and state, index-order work queue (WBC_FIFO_DISPATCH), %d steps; the timed loop replays one " \
                                      "state, so each solve's previous cost predicts this one exactly -- see --workload %s for a state that moves" % (fifo_steps, ROLLOUT)
        if sweep_stats:
            line["stats"]["sweep"] = sweep_stats
        if world == 1 and cpu_baseline and not reference_built():
            line["cpu_baseline"] = NO_CPU_BASELINE
        elif world == 1 and cpu_baseline:
            kind, tot, _ = cpu_reference_run(sc, 1, 0, min(n, 4096), env.cores)
            line["cpu_baseline"] = {"value": min(n, 4096) / tot, "unit": UNIT, "cores": env.cores, "kind": kind,
                                    "sample": "one pass over the first %d instances of the workload, all %d host threads" % (min(n, 4096), env.cores)}
        if last is not None:
            dump_outputs(dump, last)
    batch.close()
    del dev_in, dev_out, stat_out
    torch.cuda.empty_cache()
    return line


ALSO = ("trot_65536", "mixed_terrain_1m")      # the other batch configs of BASELINE.json, timed in the same run for a few steps


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == REPLAY:
        if args.impl == "reference":
            args.no_cpu_baseline = False
        return single_robot_replay(args) if rank == 0 else 0
    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, world)
    env = Env(args)
    if args.workload == ROLLOUT:
        from bench_rollout import bench_trot_rollout
        line = bench_trot_rollout(env, args)
    elif args.workload == SWEEP:
        from bench_rollout import bench_push_sweep
        line = bench_push_sweep(env, args)
    else:
        line = bench_batch(env, args, args.workload, args.steps, args.warmup, per_gpu=args.per_gpu, cpu_baseline=not args.no_cpu_baseline,
                           fifo_steps=0 if (args.no_also or args.fifo) else min(args.steps, 10), fifo=args.fifo, traj_on_device=args.traj_on_device,
                           dump=args.dump_outputs)
        if args.workload == "standing_4096" and not args.no_also and not args.fifo and args.per_gpu is None:
            also = {}
            for name in ALSO:
                l2 = bench_batch(env, args, name, min(args.steps, 5), 3, fifo_steps=min(args.steps, 3))
                if l2 is not None:
                    also[name] = {k: l2[k] for k in ("value", "unit", "ms_per_step", "p50_ms", "steps", "warmup", "e2e", "stats", "value_fifo", "dispatch_gain") if k in l2}
                    also[name]["workload"] = l2["config"]["workload"]
                    also[name]["instances_per_gpu"] = l2["config"]["instances_per_gpu"]
                    also[name]["roofline"] = {k: l2["roofline"][k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "traffic", "traffic_source", "kernel_ms", "front_kernel_ms",
                                                                              "flops_per_solve", "algorithmic_bytes_per_launch", "intermediate_bytes_per_launch") if k in l2["roofline"]}
                    also[name]["clocks"] = l2["clocks"]
            if line is not None:
                line["also"] = also
                line["also_note"] = "BASELINE.json configs[2] and configs[3] (131072 instances per GPU = 1048576 on 8 GPUs) timed in the same run, same method, fewer steps"
    if rank == 0 and line is not None:
        print(json.dumps(line))
    env.close()
    return 0


def reference_arm(args, world):
    cfg = workload_cfg(args.workload if args.workload != ROLLOUT else "standing_4096")
    n_cfg = cfg.pop("n")
    sweep = args.workload == SWEEP
    per_gpu = args.per_gpu or (n_cfg // 8 if args.workload == "mixed_terrain_1m" else (n_cfg // world if sweep else n_cfg))
    cores = os.cpu_count() or 1
    config = {"workload": "%s: %d DogBot instances per GPU x %d GPU(s), 18-DoF, mode mix %s, pushes=%s, terrain=%s, seed %d" % (
        args.workload, per_gpu, world, cfg["mode_mix"], cfg["pushes"], cfg["terrain"], cfg["seed"]),
        "instances_per_gpu": per_gpu, "global_batch": per_gpu * world, "parallelism": "shard%d" % world,
        "l2": "flushed between timed steps (256 MiB write)",
        "dispatch": "fifo" if args.fifo else "longest-first, predicted from each instance's previous cycle (results are order-independent)",
        "solver": "DENSE-AUL/QQP restatement, reference settings (1e-2, 1e4, 5)"}
    sc = S.push_sweep(n=min(per_gpu, 4096)) if sweep else S.make(per_gpu, start=0, **cfg)
    sample = per_gpu if (cores >= 16 or per_gpu <= 1024) else 1024
    sample = min(sample, 4096)
    kind, tot, times = cpu_reference_run(sc, args.steps, args.warmup, sample, cores)
    val = sample * args.steps / tot
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "first %d instances of the workload per step, all %d host threads" % (sample, cores)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
