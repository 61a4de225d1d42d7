#!/usr/bin/env python
"""One step of a bound group of 256 robots with every cycle input in GPU memory, served three ways and timed alternately
in one process.

  python scripts/time_group_device_inputs.py [--rounds 3 --steps 40 --warmup 5 --out FILE]

Fleets (configs[4] scenarios: robot r has its own heading, path and noise), all members on ONE shared device map (robot
0's 100 x 100 map as a CUDA tensor, every member in MPPI_COSTMAP_DEVICE mode):
  uniform  256 x (2000 x 56)
  mixed    128 x (2000 x 56), 64 x (1000 x 56), 64 x (1000 x 80), interleaved as in profiles/r06_mixed_group.txt

  host      mppi_optimize_batch: the host builds every member's record and uploads them (pose, path ... from host memory)
  device    mppi_optimize_group_device: the same inputs as CUDA tensors, the records built on the device
  resident  mppi_optimize_batch_resident: records uploaded beforehand, the device-only floor

Per way and round: end-to-end host time of the call with timing off (p50, p90), then its device span with timing on
(mppi_batch_span_ms, p50, p90), each over --steps steps with 256 MiB written between steps (cold L2, as bench.py).  The
device way calls the C entry point with its argument structs built once (the inputs do not change between steps), so
that the number is the library's, not the Python helper's.
"""
import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpcholonavigation_b200 import Engine, abi, load_product, scenarios  # noqa: E402

N_ROBOTS = 256
FLEETS = {"uniform": {k: (2000, 56) for k in range(4)}, "mixed": {0: (2000, 56), 1: (2000, 56), 2: (1000, 56), 3: (1000, 80)}}


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


class Fleet:
    def __init__(self, fns, shapes, torch):
        self.fns, self.n = fns, N_ROBOTS
        self.robots = [scenarios.config5_robot(r, batch=shapes[r % 4][0], steps=shapes[r % 4][1]) for r in range(self.n)]
        shared = torch.from_numpy(np.ascontiguousarray(self.robots[0].cycle.costmap)).cuda()
        self.cycles = [dataclasses.replace(sc.cycle, costmap=shared) for sc in self.robots]
        self.engines = []
        for sc in self.robots:
            e = Engine(fns, **sc.cfg)
            e.set_robot(sc.robot)
            e.set_critics(sc.critics)
            e.set_noise(*sc.noise())
            e.set_costmap_residency(True)
            self.engines.append(e)
        self.hs = (abi.H * self.n)(*[e.h for e in self.engines])
        assert fns["batch_bind"](self.hs, self.n) == 0, fns["last_error"](self.engines[0].h)
        self.ins, self.outs = (abi.CycleIn * self.n)(), (abi.CycleOut * self.n)()
        self.keep = []
        for i, (sc, c) in enumerate(zip(self.robots, self.cycles)):
            cin, k = c.pack()
            self.ins[i] = cin
            arrs = [np.empty(sc.cfg["time_steps"], np.float32) for _ in range(3)]
            self.outs[i].control_vx, self.outs[i].control_vy, self.outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
            self.keep.append((k, arrs))
        stride = max(len(c.path_x) for c in self.cycles)
        state = np.zeros((self.n, 8)); tol = np.zeros(self.n); size = np.zeros(self.n, np.int32)
        path = np.zeros((self.n, 3, stride), np.float32)
        for i, c in enumerate(self.cycles):
            state[i] = [*c.pose, *c.speed, *c.goal]
            tol[i] = c.goal_checker_xy_tolerance
            size[i] = len(c.path_x)
            path[i, :, :size[i]] = (c.path_x, c.path_y, c.path_yaw)
        self.dev_in = [torch.from_numpy(a).cuda() for a in (state, tol, size, path)]
        self.gi = abi.GroupInputs()
        self.gi.state, self.gi.goal_checker_xy_tolerance, self.gi.path_size, self.gi.path = (t.data_ptr() for t in self.dev_in)
        self.gi.path_stride = stride
        self.maps = (abi.Costmap * self.n)()
        for i, c in enumerate(self.cycles):
            self.maps[i] = self.ins[i].costmap
        torch.cuda.synchronize()
        for e, c in zip(self.engines, self.cycles):
            e.upload_cycle(c)

    def host(self):
        assert self.fns["optimize_batch"](self.hs, self.ins, self.outs, self.n) == 0, self.fns["last_error"](self.engines[0].h)

    def device(self):
        assert self.fns["optimize_group_device"](self.hs, self.n, C.byref(self.gi), self.maps, self.outs) == 0, \
            self.fns["last_error"](self.engines[0].h)

    def resident(self):
        assert self.fns["optimize_batch_resident"](self.hs, self.outs, self.n) == 0

    def span_ms(self):
        span = C.c_float(0.0)
        assert self.fns["batch_span_ms"](self.hs, self.n, C.byref(span)) == 0
        return span.value

    def set_timing(self, on):
        for e in self.engines:
            e.set_timing(on)

    def close(self):
        for e in self.engines:
            e.close()


def measure(fleet, way, steps, warmup, flush):
    call = getattr(fleet, way)
    e2e, dev = [], []
    fleet.set_timing(False)
    for _ in range(warmup):
        call()
    for _ in range(steps):
        flush()
        t0 = time.perf_counter()
        call()
        e2e.append((time.perf_counter() - t0) * 1e3)
    fleet.set_timing(True)
    for _ in range(warmup):
        call()
    for _ in range(steps):
        flush()
        call()
        dev.append(fleet.span_ms())
    return [float(np.percentile(v, q)) for v in (e2e, dev) for q in (50, 90)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the report here")
    a = ap.parse_args()
    import torch
    buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush():
        buf.zero_()
        torch.cuda.synchronize()

    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"gpu (name, power limit, sm clock, max sm clock) before: {gpu_identity()}")
    say(f"{N_ROBOTS} robots per fleet, one shared device map; cold L2 (256 MiB written between steps), {a.steps} steps per "
        f"way and round, {a.warmup} warm-up, ways alternated; times in us")
    fns = load_product()
    results = {}
    for fname, shapes in FLEETS.items():
        fleet = Fleet(fns, shapes, torch)
        for r in range(a.rounds):
            for way in ("host", "device", "resident"):
                v = measure(fleet, way, a.steps, a.warmup, flush)
                results.setdefault(f"{fname}/{way}", []).append(v)
                say(f"round {r} {fname:8s} {way:8s} e2e p50 {v[0] * 1e3:8.1f} p90 {v[1] * 1e3:8.1f}   "
                    f"device span p50 {v[2] * 1e3:8.1f} p90 {v[3] * 1e3:8.1f}")
        fleet.close()
        say(f"gpu after fleet {fname}: {gpu_identity()}")
    say("summary (median over rounds of the per-round percentiles):")
    for k, v in results.items():
        m = np.median(np.asarray(v), axis=0) * 1e3
        say(f"  {k:18s} e2e p50 {m[0]:8.1f} p90 {m[1]:8.1f}   device span p50 {m[2]:8.1f} p90 {m[3]:8.1f}")
    say(json.dumps({k: [[x * 1e3 for x in r] for r in v] for k, v in results.items()}))
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
