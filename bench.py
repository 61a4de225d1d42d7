#!/usr/bin/env python
"""bench.py -- rollout-steps/s and optimize() latency of the MPPI hot path.

  python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference] [--dump-outputs DIR]

A "step" is one Optimizer::optimize() (nav2_sortham_controller/src/optimizer.cpp:157-164) over one batch of
synthetic input: iteration_count x {noised rollout, critics, softmax update}.  Protocol = the reference's own
harness (benchmark/optimizer_benchmark.cpp:85-93): fixed robot pose, control sequence carried between cycles.

workloads (BASELINE.json configs):
  omni_1000x56        configs[0]/[1]: Omni 1000 x 56, dt 0.05, default critic set, 100x100 costmap, 40-point path,
                      reference-style injected noise.  THE headline line; at N>1 every rank runs this same problem
                      with its own noise draw (replicas, no data-path collective: weak scaling).
  obstacles_16384x56  configs[2]: 16384 x 56, 400x400 costmap, ObstaclesCritic in footprint mode.
  obstacles_dense_16384x56  the same with the robot boxed in (rectangular footprint inside a ring of discs): the footprint
                      branch is taken by ~14 % of the visited poses in every cycle (configs[2]'s literal geometry: 0.2 % of
                      the first cycle, none afterwards; cpu_baseline.footprint_branch reports the counts for both).
  sharded_262144x100  configs[3]: 262144 x 100 sharded over the ranks, Philox noise by global trajectory index,
                      two exchanges (furthest path point; softmax partials) over NVLink peer memory or NCCL (strong scaling).
  robots_256          configs[4]: 256 robots x (2000 x 56), 256/N per rank, one bound group per rank, no exchange.

Without --workload the ONE line printed is the omni_1000x56 line and it carries three nested records measured in the
same process at the same N and with the same --steps / --warmup: "obstacles_16384x56" and "obstacles_dense_16384x56" (N = 1 only), "sharded_262144x100" and "robots_256", each with
ms_per_step, e2e, per-kernel ms, roofline and a "parity" object produced in the same run (every rank's result against
the CPU oracle; "MISMATCH" makes the process exit non-zero after the line is printed).

value  = whole-job rollout-steps/s with inputs resident in HBM (mppi_upload_cycle once, then
         mppi_optimize_resident per step), timed with CUDA events on the launching stream, max over ranks,
         L2 flushed between timed steps.
e2e    = the same metric through mppi_optimize() with HOST buffers: costmap + cycle record H2D and the control
         sequence D2H inside the timed region (host wall clock per call).
roofline = the bound that binds the dominant kernel: "hbm" (algorithmic bytes / duration against MEASURED_PEAKS.json)
         or "issue" (warp instructions of that launch, from the ncu capture recorded in profiles/ncu_kernel_counters.json,
         / duration against the issue-slot peak measured by scripts/peak_microbench.cu, profiles/measured_sm_peaks.json);
         whichever fraction is larger is reported as frac, the other one beside it.

--dump-outputs DIR writes what the caller of the timed path received in its LAST timed step, for every workload of the
line, as DIR/<workload>.<array>.npy (float32 / float64): the control sequence vx, vy, wz ([T], or [robots, T] for
robots_256), fail_flag and furthest_reached_path_point (-1: none).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.
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

from mpcholonavigation_b200 import Engine, scenarios  # noqa: E402

METRIC = "rollout_steps_per_sec"
UNIT = "rollout-steps/s"
RTOL, ATOL = 1e-4, 1e-6          # north_star's parity bar on the control sequence
ZERO_COPY_MAX = 96 * 1024        # costmaps above this are handed over in place (registered caller memory)
DEFAULT_STEPS, DEFAULT_WARMUP = 1000, 20


def algorithmic_bytes(B, T, N, cells, iterations=1):
    """SURVEY.md 8(d): bytes(optimize) = iteration_count * (12 B T + 4 B) + cells + 24 T + 12 N"""
    return iterations * (12 * B * T + 4 * B) + cells + 24 * T + 12 * N


def pick_scenario(workload, rank, world):
    if workload == "omni_1000x56":
        # N > 1: every rank runs the SAME problem (configs[1]) with its own noise draw, so that the per-GPU work really is
        # fixed as N grows (weak scaling).
        sc = scenarios.config1(noise_seed=1 + rank)
        sc.name = "omni_1000x56"
        return sc, "injected"
    if workload == "obstacles_16384x56":
        return scenarios.config3(), "injected"
    if workload == "obstacles_dense_16384x56":
        # configs[2] with the robot boxed in (rectangular footprint inside a ring of discs): the footprint branch of the
        # critic is taken by ~13 % of the visited poses in every cycle; SURVEY 8d's literal geometry takes it in 0.2 % of the
        # first cycle's poses and never once the control sequence has moved away (cpu_baseline.footprint_branch has both)
        return scenarios.config3(dense=True), "injected"
    if workload == "sharded_262144x100":
        return scenarios.config4(), "philox"
    if workload == "robots_256":
        sc = scenarios.config5_robot(rank)   # CPU arm: the robots are independent and the reference runs them one by one
        return sc, "injected"
    raise SystemExit(f"unknown workload {workload}")


def make_config(workload, sc, noise_kind, world, exchange, flush):
    """The `config` object of the JSON line: a function of the workload and of N only, so that the reference arm prints the
    very same object as the GPU arm."""
    B, T = sc.cfg["batch_size"], sc.cfg["time_steps"]
    sharded = workload == "sharded_262144x100"
    if workload == "robots_256":
        n = 256 // world
        return {"workload": "robots_256", "robots": 256, "robots_per_rank": n, "batch_size": B, "time_steps": T,
                "iteration_count": 1, "critics": [c[0] for c in sc.critics], "costmap": list(sc.cycle.costmap.shape),
                "path_points": len(sc.cycle.path_x), "noise": "injected",
                "parallelism": "independent robots sharded over the ranks, one bound group per rank, no exchange",
                "l2": "cold: 256 MiB written between timed steps" if flush else "warm (no flush)"}
    in_place = sc.cycle.costmap.size > ZERO_COPY_MAX
    if sharded and world > 1:
        par = "sharded over ranks, 2 exchanges (%s)" % ("in-kernel over NVLink peer memory" if exchange == "peer"
                                                        else "NCCL all-reduce + all-gather")
    elif world > 1:
        par = "replicas: the same problem on every rank, own noise draw, no exchange"
    else:
        par = "single GPU"
    return {"workload": sc.name, "batch_size": B, "time_steps": T, "iteration_count": sc.cfg.get("iteration_count", 1),
            "critics": [c[0] for c in sc.critics], "costmap": list(sc.cycle.costmap.shape),
            "path_points": len(sc.cycle.path_x), "noise": noise_kind,
            "per_rank_batch": B // world if sharded else B,
            "costmap_memory": "registered as pinned, uploaded in place" if in_place else "staged (memcpy into pinned staging)",
            "parallelism": par,
            "l2": "cold: 256 MiB written between timed steps" if flush else "warm (no flush)"}


class ClockSampler(threading.Thread):
    """nvidia-smi's clocks line through NVML, sampled DURING the timed region."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.sm.append(int(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM)))
                mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def pct(a, q):
    return float(np.percentile(np.asarray(a, np.float64), q))


def result_outputs(r):
    """what a caller of optimize() receives (api.Result), as the arrays of --dump-outputs"""
    f = r.furthest_reached_path_point
    return {"vx": r.vx, "vy": r.vy, "wz": r.wz, "fail_flag": np.array([float(r.fail_flag)]),
            "furthest_reached_path_point": np.array([-1.0 if f is None else float(f)])}


def dump_outputs(directory, outputs):
    """--dump-outputs: DIR/<workload>.<array>.npy for every workload of the line"""
    os.makedirs(directory, exist_ok=True)
    for workload, arrays in outputs.items():
        for name, a in arrays.items():
            np.save(os.path.join(directory, f"{workload}.{name}.npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# CPU side: the reference arm and the cpu_baseline object
# ----------------------------------------------------------------------------------------------------------------
def cpu_identity():
    """pins this process to ONE core (the reference is single-threaded; BASELINE.md asks for a pinned core and the CPU
    model in the same log) and says which"""
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    core = None
    try:
        allowed = sorted(os.sched_getaffinity(0))
        core = allowed[len(allowed) // 2]      # away from core 0, which the kernel favours for interrupts
        os.sched_setaffinity(0, {core})
    except (AttributeError, OSError):
        pass
    return model, core, os.cpu_count()


def oracle_engine(sc, noise_kind, fast=True, wide=False):
    from tests import oracle_loader
    fns = oracle_loader.load(fast=fast)
    e = Engine(fns, **sc.cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise_kind == "injected":
        e.set_noise(*sc.noise())
    elif noise_kind == "philox":
        e.generate_noise(0)
    if wide:
        fns["set_wide_reductions"](e.h, 1)
    return e


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path, timed on this box's host cores.  The xtensor
    reference cannot be built offline (no rclcpp / nav2_costmap_2d / xtensor): this is the oracle port built
    with the reference's flags (oracle/Makefile, -O3 -mavx2 -mfma -ffast-math).  The reference is
    single-threaded (XTENSOR_USE_TBB 0 / XTENSOR_USE_OPENMP 0, CMakeLists.txt:7-8), so cores = 1."""
    if rank != 0:
        return
    model, core, ncpu = cpu_identity()
    sc, noise_kind = pick_scenario(args.workload, 0, 1)
    B, T = sc.cfg["batch_size"], sc.cfg["time_steps"]
    e = oracle_engine(sc, noise_kind)
    # without --steps / --warmup the sample is bounded: a step of the big configs takes seconds on one core
    est = B * T * 1.0e-7
    steps = args.steps if args.steps is not None else max(1, min(DEFAULT_STEPS, int(60.0 / max(est, 1e-6))))
    warm = args.warmup if args.warmup is not None else (DEFAULT_WARMUP if est * DEFAULT_WARMUP < 20.0
                                                        else max(1, int(20.0 / est)))
    for _ in range(warm):
        e.optimize(sc.cycle)
    lat = []
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        r = e.optimize(sc.cycle)
        lat.append((time.perf_counter() - t0) * 1e3)
    wall = time.perf_counter() - t_all
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {sc.name: result_outputs(r)})
    iters = sc.cfg.get("iteration_count", 1)
    value = B * T * iters * steps / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": wall / steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.workload in ("sharded_262144x100", "robots_256") else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args.workload, sc, noise_kind, args.gpus, args.exchange, not args.no_flush),
        "latency_ms": {"p50": pct(lat, 50), "p90": pct(lat, 90), "p99": pct(lat, 99)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "cpu_model": model, "pinned_core": core,
                         "sample": f"{steps} optimize() calls of {sc.name} on 1 host thread pinned to core {core} of {ncpu} "
                                   f"({model}), reference-flags build of the oracle port (xtensor reference not buildable offline)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def cpu_baseline(sc, noise_kind, budget_s=12.0):
    model, core, ncpu = cpu_identity()
    B, T = sc.cfg["batch_size"], sc.cfg["time_steps"]
    e = oracle_engine(sc, noise_kind)
    e.optimize(sc.cycle)
    branch_cold = footprint_branch(e, B * T)
    n, t0 = 0, time.perf_counter()
    lat = []
    while True:
        t1 = time.perf_counter()
        e.optimize(sc.cycle)
        lat.append((time.perf_counter() - t1) * 1e3)
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= 2000:
            break
    wall = time.perf_counter() - t0
    branch = footprint_branch(e, B * T)
    e.close()
    out = {"value": B * T * sc.cfg.get("iteration_count", 1) * n / wall, "unit": UNIT, "cores": 1, "kind": "port",
           "p50_ms": pct(lat, 50), "cpu_model": model, "pinned_core": core,
           "sample": f"{n} optimize() calls of {sc.name} in {wall:.1f} s on 1 host thread pinned to core {core} of {ncpu} ({model}); "
                     f"the reference is single-threaded; oracle port, reference-flags build"}
    if branch:
        out["footprint_branch"] = {"first_cycle_zero_control_sequence": branch_cold, f"cycle_{n + 1}_warm_started": branch,
                                   "note": "poses visited = poses of the batch before a trajectory's first collision (the "
                                           "critics break there); counted by the CPU oracle"}
    return out


def footprint_branch(e, poses):
    """SURVEY 8d: the fraction of poses for which the obstacle-type critics leave the point cost for the footprint check
    (cost_critic.cpp:204-209, obstacles_critic.cpp:214-220), counted by the CPU oracle in its last optimize()"""
    import ctypes as C
    if "get_counters" not in e.f:
        return None
    c = (C.c_uint64 * 4)()
    e.f["get_counters"](e.h, c)
    out = {}
    for name, visited, fp in (("CostCritic", c[0], c[1]), ("ObstaclesCritic", c[2], c[3])):
        if visited:
            out[name] = {"poses_visited": int(visited), "footprint_checks": int(fp), "fraction_of_visited": fp / visited,
                         "fraction_of_all_poses": fp / poses}
    return out or None


# ----------------------------------------------------------------------------------------------------------------
# rooflines
# ----------------------------------------------------------------------------------------------------------------
def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "hbm_src": "fallback of B200_PROFILING.md", "issue_gips": None, "fp32_tflops": None,
             "sm_src": None}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        peaks["hbm_gbs"], peaks["hbm_src"] = float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst)"
    p = os.path.join(ROOT, "profiles", "measured_sm_peaks.json")
    if os.path.exists(p):
        d = json.load(open(p))
        peaks["issue_gips"] = d.get("warp_inst_per_s_peak", 0.0) / 1e9 or None
        peaks["fp32_tflops"] = d.get("fp32_ffma_tflops")
        peaks["sm_src"] = "profiles/measured_sm_peaks.json (scripts/peak_microbench.cu on this pool's B200)"
    return peaks


def kernel_counters(kernel, B_local, T, tag=""):
    """ncu counters of ONE launch of `kernel` at this launch size (profiles/ncu_kernel_counters.json), or None; `tag`
    selects the capture of a workload variant with the same launch size ("dense:")"""
    p = os.path.join(ROOT, "profiles", "ncu_kernel_counters.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(f"{tag}{kernel}@{B_local}x{T}")


def make_roofline(kernel, dur_ms, alg_bytes, B_local, T, peaks, note, tag=""):
    """the bound that binds: HBM (algorithmic bytes) or issue slots (warp instructions from the ncu capture of this launch size)"""
    hbm = alg_bytes / (dur_ms * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": kernel, "achieved": hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": hbm / peaks["hbm_gbs"], "traffic": None, "algorithmic_bytes_per_launch": int(alg_bytes),
            "kernel_ms": dur_ms, "peak_source": peaks["hbm_src"], "note": note}
    kc = kernel_counters(kernel, B_local, T, tag)
    if kc:
        roof["traffic"] = kc.get("dram_bytes")
        roof["counters_source"] = kc.get("source")
        inst = kc.get("warp_inst")
        if inst and peaks["issue_gips"]:
            gips = inst / (dur_ms * 1e-3) / 1e9
            frac_issue = gips / peaks["issue_gips"]
            side = {"bound": "issue", "achieved": gips, "peak": peaks["issue_gips"], "unit": "G warp-inst/s",
                    "frac": frac_issue, "warp_inst_per_launch": int(inst), "peak_source": peaks["sm_src"]}
            if frac_issue > roof["frac"]:
                hbm_side = {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "peak_source")}
                roof.update(side)
                roof["hbm"] = hbm_side
            else:
                roof["issue"] = side
    return roof


def robots_roofline(roof, kc, n, step_ms, peaks):
    """adds the ncu side of the 256-robot step to its roofline: counters of ONE step of a bound group (every launch of the
    step summed, profiles/ncu_kernel_counters.json: robots_step@BxT), scaled to the n robots of this rank; the bound that
    binds is the larger fraction, as in make_roofline"""
    if not kc:
        return roof
    scale = n / kc["n_robots"]
    roof["traffic"] = int(kc["dram_bytes"] * scale)
    roof["counters_source"] = kc["source"]
    roof["traffic_note"] = (f"sum over the {kc['launches']} launches of one step of {kc['n_robots']} robots"
                            + ("" if scale == 1.0 else f", scaled by {n}/{kc['n_robots']}"))
    if peaks["issue_gips"]:
        gips = kc["warp_inst"] * scale / (step_ms * 1e-3) / 1e9
        side = {"bound": "issue", "achieved": gips, "peak": peaks["issue_gips"], "unit": "G warp-inst/s",
                "frac": gips / peaks["issue_gips"], "warp_inst_per_step": int(kc["warp_inst"] * scale),
                "peak_source": peaks["sm_src"]}
        if side["frac"] > roof["frac"]:
            hbm_side = {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "peak_source")}
            roof.update(side)
            roof["hbm"] = hbm_side
        else:
            roof["issue"] = side
    roof["per_kernel_ncu"] = {k: {"share_of_ncu_time": v["ncu_duration_us"] / max(kc["ncu_duration_us"], 1e-9),
                                  "dram_bytes": int(v["dram_bytes"] * scale), "warp_inst": int(v["warp_inst"] * scale)}
                              for k, v in kc["per_kernel"].items()}
    return roof


# ----------------------------------------------------------------------------------------------------------------
# GPU side
# ----------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, rank, world, local_rank, torch, dist, fns):
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.torch, self.dist, self.fns = torch, dist, fns
        self.flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.peaks = load_peaks()
        self.outputs = {}   # workload -> {array name: what the last timed step returned}, for --dump-outputs

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def flush_l2(self):
        if self.flush is not None:
            self.flush.zero_()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor([float(v) for v in vals], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]


def controls_deviation(got, want):
    """worst violation of |got - want| <= ATOL + RTOL |want| over the three control planes, as a multiple of the bound
    (<= 1 passes), and the largest absolute deviation for the record"""
    worst, dev = 0.0, 0.0
    for a, b in zip(got, want):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        worst = max(worst, float(np.max(np.abs(a - b) / (ATOL + RTOL * np.abs(b)))))
        dev = max(dev, float(np.max(np.abs(a - b))))
    return worst, dev


def connect_shards(ctx, e):
    """exchanges of a sharded handle: NVLink peer mailboxes (default) or NCCL"""
    import ctypes as C
    from mpcholonavigation_b200 import abi
    torch, dist, fns = ctx.torch, ctx.dist, ctx.fns
    if ctx.args.exchange == "nccl":
        uid = torch.zeros(abi.NCCL_UNIQUE_ID_BYTES, dtype=torch.uint8)
        if ctx.rank == 0:
            buf = (C.c_uint8 * abi.NCCL_UNIQUE_ID_BYTES)()
            assert fns["comm_get_unique_id"](buf) == 0
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        uid = uid.cuda()
        dist.broadcast(uid, 0)
        e.comm_init(bytes(uid.cpu().tolist()), ctx.rank, ctx.world)
    else:
        mine_h = torch.tensor(list(e.comm_mailbox_handle()), dtype=torch.uint8, device="cuda")
        all_h = [torch.zeros_like(mine_h) for _ in range(ctx.world)]
        dist.all_gather(all_h, mine_h)
        e.comm_connect_peers([bytes(t.cpu().tolist()) for t in all_h], ctx.rank, ctx.world)
        dist.barrier()


def sharded_parity(ctx, batch=65536, cycles=2):
    """In-run cross-rank check of the sharded path: config 4 at `batch` x 100 sharded over the ranks exactly like the timed
    workload (Philox by global trajectory index, both exchanges); the noise every rank drew is gathered on rank 0 and
    injected into the CPU oracle (order-free accumulators, see tests/test_gpu_parity_full.py); EVERY rank compares its own
    control sequence, fail flag and furthest reached path point with the oracle's, cycle by cycle."""
    torch, dist = ctx.torch, ctx.dist
    sc = scenarios.config4(batch=batch)
    T = sc.cfg["time_steps"]
    cfg = dict(sc.cfg)
    cfg["device"] = ctx.local_rank
    cfg["seed"] = 3
    if ctx.world > 1:
        cfg["batch_size"] = batch // ctx.world
        cfg["shard_offset"] = ctx.rank * cfg["batch_size"]
        cfg["shard_total"] = batch
    e = Engine(ctx.fns, **cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.generate_noise(0)
    if ctx.world > 1:
        connect_shards(ctx, e)
    mine = torch.from_numpy(np.stack(e.get_noise())).cuda()            # [3][B_local][T]
    if ctx.world > 1:
        parts = [torch.empty_like(mine) for _ in range(ctx.world)]
        dist.all_gather(parts, mine)
        full = torch.cat(parts, dim=1)
    else:
        full = mine
    o = None
    t_oracle = 0.0
    if ctx.rank == 0:
        noise = full.cpu().numpy()
        o = oracle_engine(sc, None, fast=False, wide=True)
        o.set_noise(noise[0], noise[1], noise[2])
    del full
    worst, worst_rel, flags_ok = 0.0, 0.0, True
    for _ in range(cycles):
        rg = e.optimize(sc.cycle)
        want = torch.zeros(3 * T + 2, dtype=torch.float64, device="cuda")
        if ctx.rank == 0:
            t0 = time.perf_counter()
            ro = o.optimize(sc.cycle)
            t_oracle += time.perf_counter() - t0
            f = -1.0 if ro.furthest_reached_path_point is None else float(ro.furthest_reached_path_point)
            want = torch.tensor(np.concatenate([ro.vx, ro.vy, ro.wz, [float(bool(ro.fail_flag)), f]]), dtype=torch.float64,
                                device="cuda")
        if ctx.world > 1:
            dist.broadcast(want, 0)
        w = want.cpu().numpy()
        wv = (w[:T].astype(np.float32), w[T:2 * T].astype(np.float32), w[2 * T:3 * T].astype(np.float32))
        dev, rel = controls_deviation((rg.vx, rg.vy, rg.wz), wv)
        worst, worst_rel = max(worst, dev), max(worst_rel, rel)
        f = -1.0 if rg.furthest_reached_path_point is None else float(rg.furthest_reached_path_point)
        flags_ok = flags_ok and float(bool(rg.fail_flag)) == w[3 * T] and f == w[3 * T + 1]
        e.set_control_sequence(*wv)
    e.close()
    if o is not None:
        o.close()
    worst, worst_rel, bad = ctx.max_over_ranks(worst, worst_rel, 0.0 if flags_ok else 1.0)
    ok = worst <= 1.0 and bad == 0.0
    return {"status": "ok" if ok else "MISMATCH", "checked": f"config 4 at {batch} x {T} sharded over {ctx.world} rank(s), "
            f"{cycles} cycles, every rank's control sequence + fail flag + furthest point against the CPU oracle on the gathered noise",
            "tolerance": f"|d| <= {ATOL} + {RTOL} |ref|", "worst_violation_ratio": worst, "max_abs_dev": worst_rel,
            "flags_equal": bad == 0.0, "oracle_s": t_oracle}


def single_parity(ctx, workload, cycles=3):
    """In-run check of a single-handle workload at its full size (N = 1 records): `cycles` optimize() calls from host
    buffers against the CPU oracle on the same injected noise - control sequence, fail flag, furthest reached path point,
    and the total cost of every trajectory; both sides continue from the oracle's control sequence."""
    sc, noise_kind = pick_scenario(workload, 0, 1)
    assert noise_kind == "injected"
    cfg = dict(sc.cfg)
    cfg["device"] = ctx.local_rank
    e = Engine(ctx.fns, **cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    e.set_noise(*sc.noise())
    o = oracle_engine(sc, "injected", fast=False)
    worst, worst_abs, worst_cost, flags_ok, t_oracle = 0.0, 0.0, 0.0, True, 0.0
    for _ in range(cycles):
        rg = e.optimize(sc.cycle)
        t0 = time.perf_counter()
        ro = o.optimize(sc.cycle)
        t_oracle += time.perf_counter() - t0
        dev, ab = controls_deviation((rg.vx, rg.vy, rg.wz), (ro.vx, ro.vy, ro.wz))
        worst, worst_abs = max(worst, dev), max(worst_abs, ab)
        cg, co = np.asarray(e.get_costs(), np.float64), np.asarray(o.get_costs(), np.float64)
        worst_cost = max(worst_cost, float(np.max(np.abs(cg - co) / (5e-6 + RTOL * np.abs(co)))))
        flags_ok = (flags_ok and bool(rg.fail_flag) == bool(ro.fail_flag)
                    and rg.furthest_reached_path_point == ro.furthest_reached_path_point)
        e.set_control_sequence(ro.vx, ro.vy, ro.wz)
    e.close()
    o.close()
    ok = worst <= 1.0 and worst_cost <= 1.0 and flags_ok
    return {"status": "ok" if ok else "MISMATCH",
            "checked": f"{sc.name} at full size, {cycles} cycles from host buffers against the CPU oracle: control sequence, "
                       "fail flag, furthest point, total cost of every trajectory",
            "tolerance": f"controls |d| <= {ATOL} + {RTOL} |ref|, costs |d| <= 5e-06 + {RTOL} |ref|",
            "worst_violation_ratio": worst, "worst_cost_violation_ratio": worst_cost, "max_abs_dev": worst_abs,
            "flags_equal": flags_ok, "oracle_s": t_oracle}


def run_workload(ctx, workload, steps, warmup, with_cpu_baseline, parity=None):
    """one workload through one handle per rank (everything but robots_256); returns the JSON object on rank 0"""
    args, rank, world, fns = ctx.args, ctx.rank, ctx.world, ctx.fns
    sharded = workload == "sharded_262144x100"
    sc, noise_kind = pick_scenario(workload, rank, world)
    cfg = dict(sc.cfg)
    cfg["device"] = ctx.local_rank
    B_total, T = cfg["batch_size"], cfg["time_steps"]
    if sharded and world > 1:
        assert B_total % world == 0
        cfg["batch_size"] = B_total // world
        cfg["shard_offset"] = rank * cfg["batch_size"]
        cfg["shard_total"] = B_total
    cfg["seed"] = 3
    e = Engine(fns, **cfg)
    e.set_robot(sc.robot)
    e.set_critics(sc.critics)
    if noise_kind == "injected":
        e.set_noise(*sc.noise())
    else:
        e.generate_noise(0)
    if sharded and world > 1:
        connect_shards(ctx, e)
    B_local = cfg["batch_size"]
    iters = cfg.get("iteration_count", 1)

    # ---- leg 1: device-resident inputs ---------------------------------------------------------
    e.upload_cycle(sc.cycle)
    for _ in range(warmup):
        e.optimize_resident()
    launches0 = e.get_profile()["kernel_launches"]
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    ctx.barrier()
    dev_ms, wall_ms = [], []
    t_region = time.perf_counter()
    for _ in range(steps):
        ctx.flush_l2()
        t0 = time.perf_counter()
        r = e.optimize_resident()
        wall_ms.append((time.perf_counter() - t0) * 1e3)
        dev_ms.append(r.device_ms)
    ctx.barrier()
    region_s = time.perf_counter() - t_region
    launches = e.get_profile()["kernel_launches"] - launches0
    ctx.outputs[workload] = result_outputs(r)

    # ---- leg 2: end to end through mppi_optimize() with host buffers ---------------------------
    # (the ctypes argument struct is marshalled once: the caller's buffers are plain host memory that does not change
    #  between cycles; every call still copies the record + costmap H2D and the result D2H inside the timed region)
    host_cycle = sc.cycle.packed()
    cm_host = host_cycle.pack()[1][3]   # the caller's costmap buffer of the packed cycle
    costmap_in_place = cm_host.nbytes > ZERO_COPY_MAX
    if costmap_in_place:
        # large costmaps are handed over in place (the controller registers Costmap2D::getCharMap() once): pinned caller
        # memory, copied H2D inside the timed region without the staging memcpy
        e.register_costmap_memory(cm_host)
    e.set_timing(False)   # the controller does not read device_ms: no event records / read-back on the production path
    for _ in range(warmup):
        e.optimize(host_cycle)
    ctx.barrier()
    e2e_ms = []
    for _ in range(steps):
        ctx.flush_l2()
        t0 = time.perf_counter()
        e.optimize(host_cycle)
        e2e_ms.append((time.perf_counter() - t0) * 1e3)
    ctx.barrier()
    e.set_timing(True)
    clocks = sampler.stop()
    prof = e.get_profile()
    h2d, d2h = prof["h2d_bytes"], prof["d2h_bytes"]

    # ---- leg 3: per-kernel durations (profiling events on), same protocol -----------------------
    e.set_profiling(True)
    e.upload_cycle(sc.cycle)
    k2, k3, xch = [], [], []
    for i in range(min(steps, 300) + 3):
        ctx.flush_l2()
        e.optimize_resident()
        p = e.get_profile()
        if i >= 3:
            k2.append(p["k2_ms"]); k3.append(p["k3_ms"]); xch.append(p["exchange_ms"])
    e.set_profiling(False)
    e.close()

    dev_total, e2e_total = ctx.max_over_ranks(float(np.sum(dev_ms)), float(np.sum(e2e_ms)))
    units = B_total * T * iters * steps if sharded else B_local * T * iters * steps * world
    if rank != 0:
        return None
    cells, N = int(sc.cycle.costmap.size), len(sc.cycle.path_x)
    alg = algorithmic_bytes(B_local, T, N, cells, iters)
    k2_ms, k3_ms, xch_ms = float(np.mean(k2)), float(np.mean(k3)), float(np.mean(xch))
    # the dominant kernel (largest share of the step) carries the roofline; the other one is reported beside it
    stream_layout = B_local >= 8192
    fused = (not stream_layout) and k3_ms == 0.0   # the library reports K3 = 0 when the fused kernel ran
    k2_name = "rollout_score_stream_kernel" if stream_layout else ("tile_fused_kernel" if fused else "rollout_score_kernel")
    k3_name = (("path_costs_tm_kernel+weighted_sums_tma_kernel (merge inside)" if world == 1 or not sharded else
                "path_costs_tm_kernel+weighted_sums_tma_kernel") if stream_layout else
               ("(fused into tile_fused_kernel)" if fused else "path_softmax_update_kernel"))
    dom_name, dom_ms, oth_name, oth_ms = (k2_name, k2_ms, k3_name, k3_ms) if k2_ms >= k3_ms else (k3_name, k3_ms, k2_name, k2_ms)
    note = ("algorithmic bytes of one optimize() (SURVEY 8d: 12 B per rollout step, noise read once) over the kernel's "
            "CUDA-event duration; " +
            ("the fused small-batch kernel reads the noise once and keeps the tile in shared memory; the config is "
             "L2-resident, single-wave and latency-bound" if fused else
             "the implementation reads the noise twice (rollout and weighted sums), so its HBM ceiling is 0.5"))
    roof = make_roofline(dom_name, dom_ms, alg, B_local, T, ctx.peaks, note, "dense:" if "dense" in workload else "")
    roof["kernel_share_of_step"] = dom_ms / max(k2_ms + k3_ms + xch_ms, 1e-9)
    roof["other_kernel"] = {"kernel": oth_name, "ms": oth_ms, "achieved": (alg / (oth_ms * 1e-3) / 1e9) if oth_ms > 0 else None}
    roof["step_achieved_gbs"] = alg / ((dev_total / steps) * 1e-3) / 1e9
    roof["step_frac_of_hbm"] = roof["step_achieved_gbs"] / ctx.peaks["hbm_gbs"]
    line = {
        "metric": METRIC, "value": units / (dev_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": dev_total / steps, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(workload, sc, noise_kind, world, args.exchange, ctx.flush is not None),
        "clocks": clocks,
        "latency_ms": {"device_p50": pct(dev_ms, 50), "device_p90": pct(dev_ms, 90), "device_p99": pct(dev_ms, 99),
                       "resident_call_p50": pct(wall_ms, 50), "e2e_p50": pct(e2e_ms, 50), "e2e_p90": pct(e2e_ms, 90),
                       "e2e_p99": pct(e2e_ms, 99)},
        "e2e": {"value": units / (e2e_total * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "p50_ms": pct(e2e_ms, 50)},
        "gpu_launches": int(launches),
        "kernels_ms": {("fused_rollout_score_update" if fused else "K2_rollout_score"): k2_ms, "K3_path_softmax_update": k3_ms,
                       "exchange_and_merge": xch_ms},
        "roofline": roof,
        "timed_region_s": region_s,
    }
    if parity is not None:
        line["parity"] = parity
    if with_cpu_baseline:
        budget = 12.0 if B_total * T <= 2_000_000 else 6.0
        line["cpu_baseline"] = cpu_baseline(pick_scenario(workload, 0, 1)[0], noise_kind, budget)
    return line


def run_robots(ctx, steps, warmup, with_cpu_baseline, check_parity):
    """configs[4]: 256 independent robots x (2000 x 56), 256 / world per rank, no data-path collective.  The rank's robots
    are one bound group (mppi_batch_bind, stream layout: one strided upload and four kernel launches per 64 robots);
    a step = every robot of the rank runs one optimize()."""
    import ctypes as C
    from mpcholonavigation_b200 import abi
    args, rank, world, fns, torch = ctx.args, ctx.rank, ctx.world, ctx.fns, ctx.torch
    n_total = 256
    assert n_total % world == 0
    n = n_total // world
    robots = [scenarios.config5_robot(rank * n + i) for i in range(n)]
    B, T = robots[0].cfg["batch_size"], robots[0].cfg["time_steps"]
    engines = []
    for sc in robots:
        cfg = dict(sc.cfg); cfg["device"] = ctx.local_rank
        e = Engine(fns, **cfg)
        e.set_robot(sc.robot); e.set_critics(sc.critics); e.set_noise(*sc.noise())
        engines.append(e)
    hs = (abi.H * n)(*[e.h for e in engines])
    # MPPI_BATCH_BIND=0: one fused launch per robot on its own stream; MPPI_BATCH_MODE=tile: the ticketed fused kernel
    # (measured alternatives, profiles/README.md)
    bound = os.environ.get("MPPI_BATCH_BIND", "1") != "0" and n > 1
    if bound:
        assert fns["batch_bind"](hs, n) == 0
    ins = (abi.CycleIn * n)()
    outs = (abi.CycleOut * n)()
    keep = []
    for i, sc in enumerate(robots):
        cin, k = sc.cycle.pack()
        ins[i] = cin
        arrs = [np.empty(T, np.float32) for _ in range(3)]
        outs[i].control_vx, outs[i].control_vy, outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
        keep.append((k, arrs))

    parity = None
    if check_parity:
        # every robot of the rank against its own CPU oracle, 2 cycles (cycle 2 from the oracle's warm start on both sides)
        t0 = time.perf_counter()
        worst, worst_rel, flags_ok = 0.0, 0.0, True
        orcs = [oracle_engine(sc, "injected", fast=False) for sc in robots]
        for _ in range(2):
            assert fns["optimize_batch"](hs, ins, outs, n) == 0
            for i, (sc, o) in enumerate(zip(robots, orcs)):
                ro = o.optimize(sc.cycle)
                dev, rel = controls_deviation(keep[i][1], (ro.vx, ro.vy, ro.wz))
                worst, worst_rel = max(worst, dev), max(worst_rel, rel)
                want = abi.UINT32_MAX if ro.furthest_reached_path_point is None else ro.furthest_reached_path_point
                flags_ok = flags_ok and bool(outs[i].fail_flag) == bool(ro.fail_flag) and outs[i].furthest_reached_path_point == want
                engines[i].set_control_sequence(ro.vx, ro.vy, ro.wz)
        for o in orcs:
            o.close()
        for e in engines:
            e.set_control_sequence(*(np.zeros(T, np.float32),) * 3)
        worst, worst_rel, bad = ctx.max_over_ranks(worst, worst_rel, 0.0 if flags_ok else 1.0)
        parity = {"status": "ok" if worst <= 1.0 and bad == 0.0 else "MISMATCH",
                  "checked": f"all {n_total} robots ({n} per rank) through mppi_optimize_batch against their own CPU oracle, 2 cycles: "
                             "control sequence, fail flag, furthest point",
                  "tolerance": f"|d| <= {ATOL} + {RTOL} |ref|", "worst_violation_ratio": worst, "max_abs_dev": worst_rel,
                  "flags_equal": bad == 0.0, "oracle_s": time.perf_counter() - t0}

    for e, sc in zip(engines, robots):
        e.upload_cycle(sc.cycle)
    span = C.c_float(0.0)
    for _ in range(warmup):
        assert fns["optimize_batch_resident"](hs, outs, n) == 0
    if bound and rank == 0:
        msg = fns["last_error"](engines[0].h)
        if msg:
            print("note:", msg.decode(), file=sys.stderr, flush=True)
    launches0 = sum(e.get_profile()["kernel_launches"] for e in engines)
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    ctx.barrier()
    dev_ms = []
    t_region = time.perf_counter()
    for _ in range(steps):
        ctx.flush_l2()
        assert fns["optimize_batch_resident"](hs, outs, n) == 0
        assert fns["batch_span_ms"](hs, n, C.byref(span)) == 0
        dev_ms.append(span.value)
    ctx.barrier()
    region_s = time.perf_counter() - t_region
    launches = sum(e.get_profile()["kernel_launches"] for e in engines) - launches0
    # copied now: the e2e leg below writes into the same output buffers
    ctx.outputs["robots_256"] = {
        **{name: np.stack([arrs[p] for _, arrs in keep]) for p, name in enumerate(("vx", "vy", "wz"))},
        "fail_flag": np.array([float(bool(o.fail_flag)) for o in outs]),
        "furthest_reached_path_point": np.array([-1.0 if o.furthest_reached_path_point == abi.UINT32_MAX
                                                 else float(o.furthest_reached_path_point) for o in outs])}
    for e in engines:
        e.set_timing(False)
    for _ in range(warmup):
        assert fns["optimize_batch"](hs, ins, outs, n) == 0
    ctx.barrier()
    e2e_ms = []
    for _ in range(steps):
        ctx.flush_l2()
        t0 = time.perf_counter()
        assert fns["optimize_batch"](hs, ins, outs, n) == 0
        e2e_ms.append((time.perf_counter() - t0) * 1e3)
    ctx.barrier()
    clocks = sampler.stop()
    h2d = sum(e.get_profile()["h2d_bytes"] for e in engines)
    d2h = sum(e.get_profile()["d2h_bytes"] for e in engines)
    for e in engines:
        e.close()
    dev_total, e2e_total = ctx.max_over_ranks(float(np.sum(dev_ms)), float(np.sum(e2e_ms)))
    units = n_total * B * T * steps
    if rank != 0:
        return None
    sc0 = robots[0]
    cells, N = int(sc0.cycle.costmap.size), len(sc0.cycle.path_x)
    alg = n * algorithmic_bytes(B, T, N, cells)
    step_ms = dev_total / steps
    tile = os.environ.get("MPPI_BATCH_MODE") == "tile"
    kname = ("rollout_score_stream_batch_kernel+path_costs_tm_batch_kernel+weighted_sums_tm_batch_kernel+merge_finalize_batch_kernel"
             if bound and not tile else ("tile_fused_batch_kernel" if bound else "tile_fused_kernel (one launch per robot)"))
    roof = make_roofline(kname, step_ms, alg, n * B, T, ctx.peaks,
                         "algorithmic bytes of the rank's robots (SURVEY 8d) over the device span of the step: first start "
                         "event to latest end event across the robots' launches (whole step, all kernels)")
    if bound and not tile:
        robots_roofline(roof, kernel_counters("robots_step", B, T), n, step_ms, ctx.peaks)
    line = {
        "metric": METRIC, "value": units / (dev_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config("robots_256", sc0, "injected", world, args.exchange, ctx.flush is not None),
        "clocks": clocks,
        "latency_ms": {"device_p50": pct(dev_ms, 50), "device_p90": pct(dev_ms, 90), "e2e_p50": pct(e2e_ms, 50),
                       "e2e_p90": pct(e2e_ms, 90), "per_robot_e2e_p50": pct(e2e_ms, 50) / n},
        "e2e": {"value": units / (e2e_total * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "p50_ms": pct(e2e_ms, 50)},
        "gpu_launches": int(launches),
        "roofline": roof,
        "timed_region_s": region_s,
    }
    if parity is not None:
        line["parity"] = parity
    if with_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(robots[0], "injected", 4.0)
    return line


_JSON_OUT = None


def _claim_stdout():
    """stdout carries the ONE JSON line: whatever native libraries print there (NCCL's version line at communicator
    creation, ...) is sent to stderr instead; emit() writes the line to the real stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    _JSON_OUT = os.fdopen(keep, "w")


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help=f"timed steps of every workload (default {DEFAULT_STEPS}; the reference arm: at most about a minute's worth)")
    ap.add_argument("--warmup", type=int, default=None,
                    help=f"untimed steps first (default {DEFAULT_WARMUP}, at least 3; the reference arm: at most about 20 s' worth)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps (steady-state number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-nested", action="store_true", help="default line only: skip the nested sharded / robots records")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="sharded workload: exchanges fused into the kernels over peer memory (default) or NCCL collectives")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of every workload returned as DIR/<workload>.<array>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup is not None:
        args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    nested = args.workload is None and not args.no_nested
    if args.workload is None:
        args.workload = "omni_1000x56"

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.steps = DEFAULT_STEPS if args.steps is None else args.steps
    args.warmup = DEFAULT_WARMUP if args.warmup is None else args.warmup

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from mpcholonavigation_b200 import load_product
    ctx = Ctx(args, rank, world, local_rank, torch, dist, load_product())
    cpu = not args.no_cpu_baseline
    failed = False

    def guarded(name, fn):
        """a nested record must never take the headline line down with it"""
        try:
            return fn()
        except Exception as exc:   # noqa: BLE001
            print(f"nested workload {name} failed: {exc!r}", file=sys.stderr, flush=True)
            return {"error": repr(exc)} if rank == 0 else None

    if args.workload == "robots_256":
        line = run_robots(ctx, args.steps, args.warmup, False, True)
    elif args.workload == "sharded_262144x100":
        line = run_workload(ctx, args.workload, args.steps, args.warmup, False, parity=sharded_parity(ctx))
    elif args.workload.startswith("obstacles_"):
        line = run_workload(ctx, args.workload, args.steps, args.warmup, False, parity=single_parity(ctx, args.workload))
    else:
        line = run_workload(ctx, args.workload, args.steps, args.warmup, False)
    extra = {}
    if nested:
        if world == 1:
            for wl in ("obstacles_16384x56", "obstacles_dense_16384x56"):
                extra[wl] = guarded(wl, lambda wl=wl: run_workload(ctx, wl, args.steps, args.warmup, False, parity=single_parity(ctx, wl)))
        extra["sharded_262144x100"] = guarded("sharded_262144x100", lambda: run_workload(
            ctx, "sharded_262144x100", args.steps, args.warmup, False, parity=sharded_parity(ctx)))
        extra["robots_256"] = guarded("robots_256", lambda: run_robots(ctx, args.steps, args.warmup, False, True))

    # the ranks part BEFORE rank 0 starts the CPU baselines: nobody spins in a collective while one host thread works
    if world > 1:
        ctx.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ctx.outputs)
    for name, rec in extra.items():
        line[name] = rec
        if isinstance(rec, dict) and (rec.get("error") or rec.get("parity", {}).get("status") == "MISMATCH"):
            failed = True
    if line.get("parity", {}).get("status") == "MISMATCH":
        failed = True
    if cpu:
        noise_kind = pick_scenario(args.workload, 0, 1)[1]
        B, T = line["config"]["batch_size"], line["config"]["time_steps"]
        line["cpu_baseline"] = cpu_baseline(pick_scenario(args.workload, 0, 1)[0], noise_kind, 12.0 if B * T <= 2_000_000 else 20.0)
        for name, rec in extra.items():
            if isinstance(rec, dict) and "error" not in rec:
                wl = "robots_256" if name == "robots_256" else name
                sc, nk = pick_scenario(wl, 0, 1)
                rec["cpu_baseline"] = cpu_baseline(sc, nk, 4.0)
    emit(line)
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
