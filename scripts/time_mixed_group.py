#!/usr/bin/env python
"""One step of a fleet of 256 robots with three shapes on one GPU, served three ways and timed alternately in one process.

  python scripts/time_mixed_group.py [--rounds 3 --steps 40 --warmup 5 --out FILE]

Fleet (configs[4] scenarios, robot r has its own map, heading and noise): 128 x (2000 x 56), 64 x (1000 x 56) and
64 x (1000 x 80), interleaved in bind order (r % 4 = 0, 1: 2000 x 56; 2: 1000 x 56; 3: 1000 x 80), so that every chunk
of 64 robots mixes all three shapes.

  mixed    the 256 robots as ONE bound group (members differ in batch_size and time_steps)
  serial   three bound groups, one per shape, stepped back to back: each mppi_optimize_batch waits for its own results
  unbound  the 256 handles unbound, through mppi_optimize_batch (one launch sequence per robot)

Per way and round: device span of mppi_optimize_batch_resident (mppi_batch_span_ms, timing on; for `serial` the sum of
the three groups' spans) and end-to-end host time of mppi_optimize_batch (inputs uploaded in the call, timing off; for
`serial` the three calls), p50 over --steps steps, 256 MiB written between steps (cold L2, as bench.py).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpcholonavigation_b200 import Engine, abi, load_product, scenarios  # noqa: E402

N_ROBOTS = 256
SHAPES = {0: (2000, 56), 1: (2000, 56), 2: (1000, 56), 3: (1000, 80)}   # by r % 4


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


class Group:
    """robots `ids` of the fleet, bound into one group or left unbound"""

    def __init__(self, fns, ids, bound):
        self.fns, self.n = fns, len(ids)
        self.robots = [scenarios.config5_robot(r, batch=SHAPES[r % 4][0], steps=SHAPES[r % 4][1]) for r in ids]
        self.engines = []
        for sc in self.robots:
            e = Engine(fns, **sc.cfg)
            e.set_robot(sc.robot)
            e.set_critics(sc.critics)
            e.set_noise(*sc.noise())
            self.engines.append(e)
        self.hs = (abi.H * self.n)(*[e.h for e in self.engines])
        if bound:
            assert fns["batch_bind"](self.hs, self.n) == 0, fns["last_error"](self.engines[0].h)
        self.ins, self.outs = (abi.CycleIn * self.n)(), (abi.CycleOut * self.n)()
        self.keep = []
        for i, sc in enumerate(self.robots):
            cin, k = sc.cycle.pack()
            self.ins[i] = cin
            arrs = [np.empty(sc.cfg["time_steps"], np.float32) for _ in range(3)]
            self.outs[i].control_vx, self.outs[i].control_vy, self.outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
            self.keep.append((k, arrs))
        for e, sc in zip(self.engines, self.robots):
            e.upload_cycle(sc.cycle)

    def resident(self):
        assert self.fns["optimize_batch_resident"](self.hs, self.outs, self.n) == 0

    def span_ms(self):
        span = C.c_float(0.0)
        assert self.fns["batch_span_ms"](self.hs, self.n, C.byref(span)) == 0
        return span.value

    def step(self):
        assert self.fns["optimize_batch"](self.hs, self.ins, self.outs, self.n) == 0

    def launches(self):
        return sum(e.get_profile()["kernel_launches"] for e in self.engines)

    def set_timing(self, on):
        for e in self.engines:
            e.set_timing(on)

    def close(self):
        for e in self.engines:
            e.close()


def measure(groups, steps, warmup, flush):
    """device span (sum over the groups, each stepped resident) and e2e (the groups stepped one after another)"""
    for _ in range(warmup):
        for g in groups:
            g.resident()
    l0 = sum(g.launches() for g in groups)
    dev = []
    for _ in range(steps):
        flush()
        total = 0.0
        for g in groups:
            g.resident()
            total += g.span_ms()
        dev.append(total)
    per_step = (sum(g.launches() for g in groups) - l0) / steps
    for g in groups:
        g.set_timing(False)
    for _ in range(warmup):
        for g in groups:
            g.step()
    e2e = []
    for _ in range(steps):
        flush()
        t0 = time.perf_counter()
        for g in groups:
            g.step()
        e2e.append((time.perf_counter() - t0) * 1e3)
    for g in groups:
        g.set_timing(True)
    msg = groups[0].fns["last_error"](groups[0].engines[0].h)
    return float(np.median(dev)), float(np.median(e2e)), per_step, (msg.decode() if msg else "")


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
    say(f"{N_ROBOTS} robots: 128 x (2000 x 56), 64 x (1000 x 56), 64 x (1000 x 80), interleaved; cold L2 (256 MiB written "
        f"between steps), {a.steps} steps per way and round, {a.warmup} warm-up, ways alternated")
    fns = load_product()
    ids = list(range(N_ROBOTS))
    ways = {
        "mixed": [Group(fns, ids, True)],
        "serial": [Group(fns, [r for r in ids if r % 4 in (0, 1)], True), Group(fns, [r for r in ids if r % 4 == 2], True),
                   Group(fns, [r for r in ids if r % 4 == 3], True)],
        "unbound": [Group(fns, ids, False)],
    }
    results = {k: [] for k in ways}
    for r in range(a.rounds):
        for name, groups in ways.items():
            dev, e2e, launches, msg = measure(groups, a.steps, a.warmup, flush)
            results[name].append((dev, e2e))
            say(f"round {r} {name:8s} device span p50 {dev * 1e3:8.1f} us   e2e p50 {e2e * 1e3:8.1f} us   "
                f"launches/step {launches:6.0f}" + (f"   ({msg})" if msg else ""))
        say(f"gpu after round {r}: {gpu_identity()}")
    say("summary (median over rounds; min .. max of the round p50s):")
    for name, v in results.items():
        d, e = np.asarray([x[0] for x in v]) * 1e3, np.asarray([x[1] for x in v]) * 1e3
        say(f"  {name:8s} device {np.median(d):8.1f} us ({d.min():.1f} .. {d.max():.1f})   "
            f"e2e {np.median(e):8.1f} us ({e.min():.1f} .. {e.max():.1f})")
    say(json.dumps({k: {"device_us": [x[0] * 1e3 for x in v], "e2e_us": [x[1] * 1e3 for x in v]} for k, v in results.items()}))
    for groups in ways.values():
        for g in groups:
            g.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
