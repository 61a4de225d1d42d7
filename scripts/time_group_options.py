#!/usr/bin/env python
"""One step of 256 robots x (2000 x 56) on one GPU when the robots run with iteration_count = 2 or regenerate_noises,
for two builds of the library loaded into the same process and timed alternately.

  python scripts/time_group_options.py PARENT.so CHANGE.so [--rounds 3 --steps 40 --warmup 5 --out FILE]

Fleets (each 256 robots, configs[4] scenarios):
  ref      iteration_count 1, bound group (what bench.py's robots_256 times)
  iter2    iteration_count 2, bound group (a build without batched iterations runs the members one by one)
  regen    regenerate_noises, bound group (skipped for a build that refuses to bind such handles)
  regen_u  regenerate_noises, unbound handles through mppi_optimize_batch (one launch sequence per robot)
Per fleet and round: device span of mppi_optimize_batch_resident (mppi_batch_span_ms, timing on) and end-to-end host
time of mppi_optimize_batch (inputs uploaded in the call, timing off), p50 over --steps steps, 256 MiB written between
steps (cold L2, as bench.py).  For unbound regenerate_noises handles the span ends behind each robot's redraw; for a
bound group it ends at the last chunk's results, ahead of the group's redraw.
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


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


class Fleet:
    def __init__(self, fns, bound, **kw):
        self.fns = fns
        self.robots = [scenarios.config5_robot(r) for r in range(N_ROBOTS)]
        T = self.robots[0].cfg["time_steps"]
        self.engines = []
        for sc in self.robots:
            e = Engine(fns, **{**sc.cfg, **kw})
            e.set_robot(sc.robot)
            e.set_critics(sc.critics)
            if kw.get("regenerate_noises"):
                e.generate_noise(5)
            else:
                e.set_noise(*sc.noise())
            self.engines.append(e)
        self.hs = (abi.H * N_ROBOTS)(*[e.h for e in self.engines])
        self.ok = not bound or fns["batch_bind"](self.hs, N_ROBOTS) == 0
        self.note = "" if self.ok else fns["last_error"](self.engines[0].h).decode()
        self.ins, self.outs = (abi.CycleIn * N_ROBOTS)(), (abi.CycleOut * N_ROBOTS)()
        self.keep = []
        for i, sc in enumerate(self.robots):
            cin, k = sc.cycle.pack()
            self.ins[i] = cin
            arrs = [np.empty(T, np.float32) for _ in range(3)]
            self.outs[i].control_vx, self.outs[i].control_vy, self.outs[i].control_wz = (a.ctypes.data_as(abi.f32p) for a in arrs)
            self.keep.append((k, arrs))
        if self.ok:
            for e, sc in zip(self.engines, self.robots):
                e.upload_cycle(sc.cycle)

    def launches(self):
        return sum(e.get_profile()["kernel_launches"] for e in self.engines)

    def measure(self, steps, warmup, flush):
        fns, hs, n = self.fns, self.hs, N_ROBOTS
        span = C.c_float(0.0)
        for _ in range(warmup):
            assert fns["optimize_batch_resident"](hs, self.outs, n) == 0
        msg = fns["last_error"](self.engines[0].h)
        l0 = self.launches()
        dev = []
        for _ in range(steps):
            flush()
            assert fns["optimize_batch_resident"](hs, self.outs, n) == 0
            assert fns["batch_span_ms"](hs, n, C.byref(span)) == 0
            dev.append(span.value)
        per_step = (self.launches() - l0) / steps
        for e in self.engines:
            e.set_timing(False)
        for _ in range(warmup):
            assert fns["optimize_batch"](hs, self.ins, self.outs, n) == 0
        e2e = []
        for _ in range(steps):
            flush()
            t0 = time.perf_counter()
            assert fns["optimize_batch"](hs, self.ins, self.outs, n) == 0
            e2e.append((time.perf_counter() - t0) * 1e3)
        for e in self.engines:
            e.set_timing(True)
        return float(np.median(dev)), float(np.median(e2e)), per_step, (msg.decode() if msg else "")

    def close(self):
        for e in self.engines:
            e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("parent")
    ap.add_argument("change")
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
    say(f"{N_ROBOTS} robots x (2000 x 56), cold L2 (256 MiB written between steps), {a.steps} steps per fleet and round, "
        f"{a.warmup} warm-up, builds alternated")
    fleets = {"ref": (True, {}), "iter2": (True, {"iteration_count": 2}),
              "regen": (True, {"regenerate_noises": 1, "seed": 11}), "regen_u": (False, {"regenerate_noises": 1, "seed": 11})}
    builds = {"parent": load_product(os.path.abspath(a.parent)), "change": load_product(os.path.abspath(a.change))}
    made = {}
    for fname, (bound, kw) in fleets.items():
        for bname, fns in builds.items():
            f = Fleet(fns, bound, **kw)
            if not f.ok:
                say(f"{fname:8s} {bname:7s} not run: {f.note}")
                f.close()
                continue
            made[(fname, bname)] = f
    results = {k: [] for k in made}
    for r in range(a.rounds):
        for key, f in made.items():
            dev, e2e, launches, msg = f.measure(a.steps, a.warmup, flush)
            results[key].append((dev, e2e))
            say(f"round {r} {key[0]:8s} {key[1]:7s} device span p50 {dev * 1e3:8.1f} us   e2e p50 {e2e * 1e3:8.1f} us   "
                f"launches/step {launches:6.0f}" + (f"   ({msg})" if msg else ""))
        say(f"gpu after round {r}: {gpu_identity()}")
    say("summary (median over rounds; min .. max of the round p50s):")
    for key, v in results.items():
        d, e = np.asarray([x[0] for x in v]) * 1e3, np.asarray([x[1] for x in v]) * 1e3
        say(f"  {key[0]:8s} {key[1]:7s} device {np.median(d):8.1f} us ({d.min():.1f} .. {d.max():.1f})   "
            f"e2e {np.median(e):8.1f} us ({e.min():.1f} .. {e.max():.1f})")
    say(json.dumps({f"{k[0]}/{k[1]}": {"device_us": [x[0] * 1e3 for x in v], "e2e_us": [x[1] * 1e3 for x in v]}
                    for k, v in results.items()}))
    for f in made.values():
        f.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
